"""Scenes lit by an environment (path_mis with env_sampling): a generated HDR sky with a small sun, and the "sun studio" built on
scenes.studio_scene's geometry.  Used by tests/test_env_sampling.py and tools/env_sampling_bench.py."""
import math

import numpy as np

import pykazen as pk
import scenes


def st_to_dir(s, t):
    """the inverse of kz_tex_eval_tree's lat-long lookup (float64): s = atan2(-x, z) / 2pi + 0.5, t = 0.5 - atan2(y, hypot(z, -x)) / pi"""
    phi = (np.asarray(s, np.float64) - 0.5) * 2 * np.pi
    lam = (0.5 - np.asarray(t, np.float64)) * np.pi
    return np.stack([-np.cos(lam) * np.sin(phi), np.sin(lam), np.cos(lam) * np.cos(phi)], -1)


def sun_sky(width=256, height=128, sun_dir=(-0.5, 0.7, -0.45), sun_deg=4.0, sun_radiance=4.0e4, sky=(0.35, 0.45, 0.7)):
    """(height, width, 3) float32 lat-long HDR: a dim sky gradient and a sun disk of angular diameter `sun_deg` (its texels' centres)"""
    t, s = np.meshgrid((np.arange(height) + 0.5) / height, (np.arange(width) + 0.5) / width, indexing="ij")
    d = st_to_dir(s, t)
    up = np.clip(d[..., 1], 0, 1)[..., None]
    img = np.asarray(sky, np.float64) * (0.15 + 0.85 * up) + 0.05
    sd = np.asarray(sun_dir, np.float64); sd /= np.linalg.norm(sd)
    cosang = d @ sd
    img[cosang >= math.cos(math.radians(sun_deg / 2))] = sun_radiance * np.array([1.0, 0.9, 0.75])
    return img.astype(np.float32)


def sky_background(sb, img, intensity=1.0):
    """background -> imagetexture (linear, as an HDR file decodes)"""
    sb.background = sb.tex_background(intensity, sb.tex_image(img, scale=1.0, srgb=False))
    return sb.background


def sun_studio(width=64, height=48, spp=65536, regularization=False, emitters=True, env_sampling=False, sky=None, max_depth=5):
    """studio_scene's ball and backdrop under a generated sun sky, plus diffuse, normal-mapped, rough-conductor, mirror and dielectric
    spheres, one visible and one invisible emitter (emitters=False: none); independent sampler of `spp` sample indices"""
    sb = pk.SceneBuilder()
    base = scenes.studio_scene(width, height, 1)
    # ball (kiss) and backdrop (diffuse) of the studio; its invisible light-panel array is replaced below
    for k in range(2):
        m = base.meshes[k]
        n = m.n_vertices
        P = np.ctypeslib.as_array(m.positions, shape=(n * 3,)).copy()
        F = np.ctypeslib.as_array(m.indices, shape=(m.n_triangles * 3,)).copy()
        N = np.ctypeslib.as_array(m.normals, shape=(n * 3,)).copy() if m.normals else None
        U = np.ctypeslib.as_array(m.uvs, shape=(n * 2,)).copy() if m.uvs else None
        b = base.bsdfs[m.bsdf]
        if b.type == pk.BSDF_KISS:
            mat = sb.bsdf_kiss(sb.tex_constant((0.871, 0.376, 0.0)), sb.tex_constant((0.3, 0, 0)), sb.tex_constant((0.0, 0, 0)), clearcoat=0.3)
        else:
            mat = sb.bsdf_diffuse((0.45, 0.45, 0.42))
        sb.mesh(P, F, mat, normals=N, uvs=U)
    rng = np.random.default_rng(5)
    nm = np.zeros((16, 16, 3), np.float32)
    nm[..., 0] = 0.5 + 0.2 * rng.uniform(-1, 1, (16, 16)); nm[..., 1] = 0.5 + 0.2 * rng.uniform(-1, 1, (16, 16)); nm[..., 2] = 0.95
    mats = [sb.bsdf_diffuse((0.7, 0.2, 0.2)), sb.bsdf_normalmap(sb.tex_image(nm, scale=3.0, srgb=False), sb.bsdf_diffuse((0.2, 0.6, 0.3))),
            sb.bsdf_roughconductor(0.25, "Cu"), sb.bsdf_mirror(), sb.bsdf_dielectric()]
    for k, mat in enumerate(mats):
        P, N, UV, F = scenes.uv_sphere((-2.0, 0.35, -1.2 + 0.6 * k), 0.28, nu=20, nv=10)
        sb.mesh(P, F, mat, normals=N, uvs=UV)
    if emitters:
        white = sb.bsdf_diffuse((0.5, 0.5, 0.5))
        # the invisible one stands at the +z edge of the backdrop, where the sun casts its shadow past the floor: a shadow ray steps through
        # an invisible emitter while a BSDF-sampled ray ends on it (integrator.cpp:259-278 vs 322-327), so where the sun is seen through one,
        # environment sampling and the reference estimator estimate different sums (DESIGN.md §3 "The environment as a light")
        P, F = scenes.orient(*scenes.quad((-1.5, 0.8, 7.8), (-0.5, 0.8, 7.8), (-0.5, 1.6, 7.8), (-1.5, 1.6, 7.8)), (-1.0, 1.2, 0.0), away=False)
        sb.mesh(P, F, white, light=sb.light((40.0, 37.0, 30.0), primary_visibility=False))
        P, F = scenes.orient(*scenes.quad((2.0, 1.0, 2.0), (2.0, 1.0, 2.8), (2.0, 1.8, 2.8), (2.0, 1.8, 2.0)), (0.0, 1.0, 2.4), away=False)
        sb.mesh(P, F, white, light=sb.light((3.0, 3.0, 4.0), primary_visibility=True))
    sky_background(sb, sun_sky() if sky is None else sky)
    sb.set_camera(width, height, 49.13434207760448, np.ctypeslib.as_array(base.camera.camera_to_world).reshape(4, 4).copy(), near=0.1, far=100.0)
    sb.set_sampler("independent", spp)
    sb.set_filter("gaussian")
    sb.set_integrator(max_depth=max_depth, regularization=regularization, env_sampling=env_sampling)
    return sb


def resolve(frame, border):
    """rgb of a bordered (H+2b, W+2b, 4) frame (block.cpp:39-45)"""
    f = np.asarray(frame, np.float64)[border:frame.shape[0] - border, border:frame.shape[1] - border]
    w = f[..., 3:4]
    return np.where(w != 0, f[..., :3] / np.where(w != 0, w, 1), 0.0)
