"""Texture filtering in path_mis (kz_integrator_desc::texture_filtering, kz_texlod.h, kz_image_filtered in kz_shade.h).

CPU: the host's camera constants equal a float64 restatement of pbrt-v4's FindMinimumDifferentials; the host-compiled footprint body
equals a float64 restatement of Approximate_dp_dxy + the barycentric Jacobian, stays finite on degenerate input and scales as geometry
says it must; the filtered lookup is level 0 when magnified, a level's bicubic at integer lambda, the lerp in between and the top level
beyond; the upload decides when filtering counts and refuses pyramids beyond 2^32 texels; the C++ host parses textureFiltering.
GPU: both probes match the host emulation; the resident pyramid is the one kzgpu_image_lookup builds; without a counted image, and with
only magnified textures, the frame is unchanged (to the float rounding of the frame's atomic sums) and so are the counters; a minified
checker converges far faster; the footprint follows the camera; two devices render like one."""
import math
import os

import numpy as np
import pytest

import pykazen as pk
import scenes


@pytest.fixture(scope="module")
def tf():
    import texfilter_emu
    texfilter_emu.build()
    return texfilter_emu


# ------------------------------------------------------------------------------------------------ numpy restatements
def lod_numpy(cam):
    """FindMinimumDifferentials (float64): (camera_from_world rows 0-2, candidates (lengths, vectors) for x and y)"""
    S = np.array(cam.sample_to_camera[:], np.float32).astype(np.float64).reshape(4, 4)
    W, H = cam.width, cam.height

    def film_dir(fx, fy):
        x, y = fx / W, fy / H
        r = [S[i, 0] * x + S[i, 1] * y + S[i, 3] for i in range(4)]
        d = np.stack([r[0] / r[3], r[1] / r[3], r[2] / r[3]], -1)
        n = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])
        return d / n[:, None]
    i = np.arange(512, dtype=np.float64)
    fx, fy = i / 511 * W, i / 511 * H
    d, rx, ry = film_dir(fx, fy), film_dir(fx + 1.0, fy), film_dir(fx, fy + 1.0)
    sign = np.copysign(1.0, d[:, 2])
    a = -1.0 / (sign + d[:, 2])
    b = d[:, 0] * d[:, 1] * a
    X = np.stack([1.0 + sign * (d[:, 0] * d[:, 0]) * a, sign * b, -sign * d[:, 0]], -1)
    Y = np.stack([b, sign + (d[:, 1] * d[:, 1]) * a, -d[:, 1]], -1)
    out = []
    for r in (rx, ry):
        dot = lambda u: r[:, 0] * u[:, 0] + r[:, 1] * u[:, 1] + r[:, 2] * u[:, 2]
        l = np.stack([dot(X), dot(Y), dot(d)], -1)
        ln = np.sqrt(l[:, 0] * l[:, 0] + l[:, 1] * l[:, 1] + l[:, 2] * l[:, 2])
        v = np.stack([l[:, 0] / ln, l[:, 1] / ln, l[:, 2] / ln - 1.0], -1)
        out.append((np.sqrt((v * v).sum(-1)), v))
    c2w = np.array(cam.camera_to_world[:], np.float32).astype(np.float64).reshape(4, 4)
    return np.linalg.inv(c2w)[:3].reshape(-1), out


def footprint_numpy(cases):
    """Approximate_dp_dxy + the triangle's barycentric Jacobian (float64) per case row of texfilter_emu.footprint"""
    c = np.asarray(cases, np.float32).astype(np.float64)
    M = c[:, :12].reshape(-1, 3, 4); ddx, ddy, s = c[:, 12:15], c[:, 15:18], c[:, 18]
    C2W = c[:, 19:35].reshape(-1, 4, 4)[:, :3, :3]
    p, n, p0, p1, p2 = (c[:, 35 + 3 * k:38 + 3 * k] for k in range(5))
    uv0, uv1, uv2 = c[:, 50:52], c[:, 52:54], c[:, 54:56]
    pc = np.einsum("nij,nj->ni", M[:, :, :3], p) + M[:, :, 3]
    nc = np.einsum("nji,nj->ni", C2W, n)
    frm = pc / np.linalg.norm(pc, axis=1, keepdims=True)
    ex, ey, ez = np.eye(3)
    refl = np.where((np.abs(frm[:, 0]) < 0.72)[:, None], ex, np.where((np.abs(frm[:, 1]) < 0.72)[:, None], ey, ez))
    u, v = refl - frm, refl - ez
    uu, vv, uv = (u * u).sum(1), (v * v).sum(1), (u * v).sum(1)
    R = (np.eye(3)[None] - (2 / uu)[:, None, None] * u[:, :, None] * u[:, None, :] - (2 / vv)[:, None, None] * v[:, :, None] * v[:, None, :]
         + (4 * uv / (uu * vv))[:, None, None] * v[:, :, None] * u[:, None, :])
    pz, nz = np.einsum("nij,nj->ni", R, pc), np.einsum("nij,nj->ni", R, nc)
    d = nz[:, 2] * pz[:, 2]
    e1, e2 = p1 - p0, p2 - p0
    g11, g12, g22 = (e1 * e1).sum(1), (e1 * e2).sum(1), (e2 * e2).sum(1)
    with np.errstate(all="ignore"):
        inv_det = 1 / (g11 * g22 - g12 * g12)
        inv_det = np.where(np.isfinite(inv_det), inv_det, 0.0)
        res = []
        for dd in (ddx, ddy):
            r = dd + ez
            t = d / (nz * r).sum(1)
            o = np.einsum("nji,nj->ni", R, t[:, None] * r - pz)
            dp = s[:, None] * np.einsum("nij,nj->ni", C2W, o)
            r1, r2 = (e1 * dp).sum(1), (e2 * dp).sum(1)
            b1, b2 = (g22 * r1 - g12 * r2) * inv_det, (g11 * r2 - g12 * r1) * inv_det
            duv = b1[:, None] * (uv1 - uv0) + b2[:, None] * (uv2 - uv0)
            res.append(np.where(np.isfinite(duv), np.clip(duv, -1e8, 1e8), 0.0))
    return np.concatenate([res[0], res[1]], 1)[:, [0, 1, 2, 3]]


def camera(fov, w, h, origin, target, thinlens=None, up=(0, 1, 0)):
    return pk.fill_camera(pk.CameraDesc(), w, h, fov, pk.lookat(origin, target, up), 1e-3, 1e4, thinlens)


# ------------------------------------------------------------------------------------------------ CPU
CAMERAS = [(fov, w, h, tl) for fov in (20.0, 45.0, 90.0) for (w, h) in ((64, 64), (1920, 1080), (300, 700)) for tl in (None, (0.05, 4.0))]


@pytest.mark.parametrize("fov,w,h,thinlens", CAMERAS)
def test_minimum_differentials_match_pbrt_loop(tf, fov, w, h, thinlens):
    cam = camera(fov, w, h, (1.0, 2.0, -3.0), (0.2, 0.1, 0.5), thinlens)
    for spp in (1, 4, 64, 1000):
        got = tf.lod(cam, spp)
        cfw, cands = lod_numpy(cam)
        np.testing.assert_allclose(got[:12], cfw, rtol=1e-6, atol=1e-6)
        for k, (lens, vecs) in enumerate(cands):
            g = got[12 + 3 * k:15 + 3 * k].astype(np.float64)
            m = lens.min()
            assert abs(np.linalg.norm(g) - m) <= 1e-5 * m
            # pbrt keeps the first strictly shorter one; points whose lengths tie in exact arithmetic (symmetric film corners) may
            # round either way, so the host's choice must be one of the shortest
            tied = vecs[lens <= m * (1 + 1e-9)]
            assert (np.linalg.norm(tied - g, axis=1) <= 1e-5 * m).any()
        assert got[18] == np.float32(max(0.125, 1 / math.sqrt(spp)))


def _random_cases(n, seed, with_uv):
    rng = np.random.default_rng(seed)
    rows = []
    while len(rows) < n:
        o = rng.uniform(-5, 5, 3); t = o + rng.normal(size=3) * 3
        if np.linalg.norm(t - o) < 0.5:
            continue
        cam = camera(rng.uniform(15, 100), int(rng.integers(32, 2000)), int(rng.integers(32, 2000)), o, t, (0.05, 3.0) if rng.random() < 0.5 else None)
        lod = None
        for _ in range(64):
            c = t + rng.normal(size=3) * 0.5
            P = (c + rng.normal(size=(3, 3)) * rng.uniform(0.05, 2.0)).astype(np.float32)
            e1, e2 = P[1] - P[0], P[2] - P[0]
            cr = np.cross(e1.astype(np.float64), e2)
            if np.linalg.norm(cr) < 0.2 * np.linalg.norm(e1) * np.linalg.norm(e2):
                continue                                  # well-shaped triangles: the Gram system is well conditioned
            b = rng.dirichlet((1, 1, 1))
            p = (np.float32(b[0]) * P[0] + np.float32(b[1]) * P[1] + np.float32(b[2]) * P[2]).astype(np.float32)
            nrm = (cr / np.linalg.norm(cr)).astype(np.float32)
            view = p - o
            if abs(np.dot(view, nrm)) < 0.2 * np.linalg.norm(view):
                continue                                  # not grazing: the plane intersection is well conditioned
            uv = rng.uniform(-2, 2, (3, 2)).astype(np.float32) if with_uv else np.array([[0, 0], [1, 0], [0, 1]], np.float32)
            if lod is None:
                lod = tf_lib.lod(cam, int(rng.choice([1, 4, 16, 64, 256])))
            rows.append(np.concatenate([lod, np.array(cam.camera_to_world[:], np.float32), p, nrm, P.reshape(-1), uv.reshape(-1)]))
            if len(rows) >= n:
                break
    return np.array(rows, np.float32)


tf_lib = None


@pytest.mark.parametrize("with_uv", [True, False])
def test_footprint_matches_numpy(tf, with_uv):
    global tf_lib
    tf_lib = tf
    cases = _random_cases(12000, 7 + with_uv, with_uv)
    got, want = tf.footprint(cases).astype(np.float64), footprint_numpy(cases)
    scale = np.maximum(np.linalg.norm(want, axis=1, keepdims=True), 1e-30)
    err = np.abs(got - want) / scale
    assert err.max() <= 1e-4, (err.max(), np.argmax(err.max(1)))
    assert (np.linalg.norm(want, axis=1) > 0).all()


def test_footprint_degenerate_inputs_stay_finite(tf):
    cam = camera(40.0, 64, 64, (0, 0, -4), (0, 0, 0))
    lod = tf.lod(cam, 1)
    c2w = np.array(cam.camera_to_world[:], np.float32)
    row = lambda p, n, P, uv: np.concatenate([lod, c2w, p, n, np.asarray(P, np.float32).reshape(-1), np.asarray(uv, np.float32).reshape(-1)])
    uv = [[0, 0], [1, 0], [0, 1]]
    quad = [[-1, -1, 0], [1, -1, 0], [-1, 1, 0]]
    cases = [
        row([0, 0, 0], [0, 0, -1], [[0, 0, 0], [1, 0, 0], [2, 0, 0]], uv),           # collinear: singular Gram system
        row([0, 0, 0], [0, 0, -1], [[0, 0, 0]] * 3, uv),                             # a point
        row([0, 0, 0], [1, 0, 0], [[0, -1, -1], [0, 1, -1], [0, -1, 1]], uv),        # the plane holds the view ray: edge-on
        row([0, 0, 0], [0, 0, 0], quad, uv),                                         # zero normal
        row([0, 0, -4], [0, 0, -1], quad, uv),                                       # the point is the camera
        row([0, 0, 0], [0, 0, -1], [[-1e-20, 0, 0], [1e-20, 0, 0], [0, 1e-20, 0]], uv),   # vanishing triangle
        row([0, 0, 0], [0, 0, -1], quad, [[0, 0], [1e30, 0], [0, 1e30]]),            # huge uv scale: clamped
    ]
    got = tf.footprint(np.array(cases, np.float32))
    assert np.isfinite(got).all() and (np.abs(got) <= 1e8).all(), got
    assert (np.abs(got[-1]) == 1e8).any()


def _fronto_lambda(tf, dist, scale=1.0, spp=1, w=512, h=512):
    """lambda at the centre of a fronto-parallel uv quad (side 2) at `dist` in front of a 45 degree camera"""
    cam = camera(45.0, 256, 256, (0, 0, 0), (0, 0, 1))
    lod = tf.lod(cam, spp)
    P = np.array([[-1, -1, dist], [1, -1, dist], [-1, 1, dist]], np.float32)
    row = np.concatenate([lod, np.array(cam.camera_to_world[:], np.float32), [0, 0, dist], [0, 0, -1], P.reshape(-1), [0, 0, 0.5, 0, 0, 0.5]]).astype(np.float32)
    d = tf.footprint(row[None])[0]
    dst = np.array([scale * d[0], -scale * d[1], scale * d[2], -scale * d[3]], np.float32)
    return float(tf.lam(w, h, dst[None])[0])


def test_footprint_geometry(tf):
    base = _fronto_lambda(tf, 3.0)
    assert abs(_fronto_lambda(tf, 6.0) - base - 1) <= 1e-3
    assert abs(_fronto_lambda(tf, 3.0, scale=2.0) - base - 1) <= 1e-3
    assert abs(_fronto_lambda(tf, 3.0, spp=64) - base + 3) <= 1e-3


def box_pyramid(img):
    """k_mip_level's 2x2 box levels in float32, same operation order"""
    levels = [np.asarray(img, np.float32)]
    while levels[-1].shape[0] > 1 or levels[-1].shape[1] > 1:
        c = levels[-1]; sh, sw = c.shape[:2]; dh, dw = max(1, sh // 2), max(1, sw // 2)
        y0 = np.minimum(2 * np.arange(dh), sh - 1); y1 = np.minimum(2 * np.arange(dh) + 1, sh - 1)
        x0 = np.minimum(2 * np.arange(dw), sw - 1); x1 = np.minimum(2 * np.arange(dw) + 1, sw - 1)
        a, b, cc, d = c[y0][:, x0], c[y0][:, x1], c[y1][:, x0], c[y1][:, x1]
        levels.append((np.float32(0.25) * (((a + b) + cc) + d)).astype(np.float32))
    return levels


def test_filtered_lookup_levels(tf):
    rng = np.random.default_rng(3)
    levels = box_pyramid(rng.uniform(0, 1, (32, 64, 3)).astype(np.float32))
    top = len(levels) - 1
    st = rng.uniform(-1, 2, (5000, 2)).astype(np.float32)
    l0 = tf.bicubic(levels, st, 0)
    for lam in (0.0, -0.5, -30.0):
        assert tf.filtered(levels, st, np.full(len(st), lam)).tobytes() == l0.tobytes()
    for l in range(1, top + 1):
        assert tf.filtered(levels, st, np.full(len(st), float(l))).tobytes() == tf.bicubic(levels, st, l).tobytes()
    lam = rng.uniform(0.01, top - 0.01, len(st)).astype(np.float32)
    lo = np.floor(lam).astype(int)
    want = np.zeros((len(st), 3))
    for l in range(top):
        sel = lo == l
        a, b = tf.bicubic(levels, st[sel], l).astype(np.float64), tf.bicubic(levels, st[sel], l + 1).astype(np.float64)
        f = (lam[sel] - l).astype(np.float64)[:, None]
        want[sel] = (1 - f) * a + f * b
    np.testing.assert_allclose(tf.filtered(levels, st, lam), want, rtol=1e-6, atol=1e-6)
    for lam in (float(top), top + 0.5, 100.0):
        assert tf.filtered(levels, st, np.full(len(st), lam)).tobytes() == tf.bicubic(levels, st, top).tobytes()


def test_lambda_is_pbrt_trilinear_level(tf):
    rng = np.random.default_rng(5)
    dst = (rng.normal(size=(10000, 4)) * 10.0 ** rng.uniform(-6, 1, (10000, 1))).astype(np.float32)
    for w, h in ((512, 512), (64, 32), (7, 300)):
        a = np.abs(dst.astype(np.float64))
        want = np.log2(np.maximum(2 * np.max(np.stack([a[:, 0] * w, a[:, 1] * h, a[:, 2] * w, a[:, 3] * h]), 0), 1e-8))
        np.testing.assert_allclose(tf.lam(w, h, dst), want, rtol=1e-5, atol=1e-5)


def _layout_scene(kind, filtering=True, integrator="path_mis"):
    sb = pk.SceneBuilder()
    img = np.zeros((16, 32, 3), np.float32)
    P = np.array([[-1, -1, 0], [1, -1, 0], [1, 1, 0]], np.float32); F = np.array([[0, 1, 2]], np.uint32)
    const = sb.tex_constant((0.5, 0.5, 0.5))
    if kind == "constants":
        b = sb.bsdf_kiss(const, const, const)
    elif kind == "background_only":
        b = sb.bsdf_kiss(const, const, const); sb.background = sb.tex_background(1.0, sb.tex_image(img))
    elif kind == "kiss_metallic":
        b = sb.bsdf_kiss(const, const, sb.tex_image(img))
    elif kind == "lambertian":
        b = sb.bsdf_lambertian(sb.tex_image(img))
    elif kind == "ggx_ramp":
        b = sb.bsdf_ggx(sb.tex_colorramp(0.1, 0.9, sb.tex_image(img)))
    elif kind == "normal_map":
        b = sb.bsdf_normalmap(sb.tex_image(img), sb.bsdf_diffuse())
    elif kind == "blend_mask":
        b = sb.bsdf_kiss(sb.tex_blend("mix", sb.tex_image(img), const, const), const, const)
    elif kind == "emitter_only":       # an emitter's BSDF is never shaded
        b = sb.bsdf_lambertian(sb.tex_image(img))
        sb.mesh(P, F, b, light=sb.light((1, 1, 1)))
        b = sb.bsdf_diffuse()
    sb.mesh(P, F, b)
    sb.set_integrator(kind=integrator, texture_filtering=filtering)
    return sb


LAYOUT = {"constants": False, "background_only": False, "kiss_metallic": True, "lambertian": True, "ggx_ramp": True, "normal_map": True,
          "blend_mask": True, "emitter_only": False}


@pytest.mark.parametrize("kind", sorted(LAYOUT))
def test_when_filtering_counts(tf, kind):
    sb = _layout_scene(kind)
    counts, total, levels = tf.layout(sb.desc())
    assert counts == LAYOUT[kind]
    n_images = len(sb.images)
    if counts:
        assert list(levels) == [5] * n_images                        # 32x16 -> 16x8 -> 8x4 -> 4x2 -> 2x1 -> 1x1
        assert total == n_images * (512 + 128 + 32 + 8 + 2 + 1)
    else:
        assert total == n_images * 512 and not levels.any()
    for off in (_layout_scene(kind, filtering=False), _layout_scene(kind, integrator="ao")):
        assert tf.layout(off.desc())[0] is False


def test_pyramid_atlas_limit(tf):
    """level 0 fits 2^32 texels, the pyramids do not: the upload refuses the scene with a clear message (image arrays are not read)"""
    sb = _layout_scene("lambertian")
    dummy = np.zeros(3, np.float32)
    sb.images[0] = pk.ImageDesc(49152, 49152, dummy.ctypes.data_as(pk.c_float_p))
    sb.bsdf_lambertian(sb.tex_image(np.zeros((1, 1, 3), np.float32)))
    sb.images[1] = pk.ImageDesc(32768, 32768, dummy.ctypes.data_as(pk.c_float_p))
    assert tf.layout(_with_images(_layout_scene("lambertian", filtering=False), sb.images).desc())[0] is False
    with pytest.raises(RuntimeError, match="mip pyramids .* larger than 2\\^32 texels"):
        tf.layout(sb.desc())


def _with_images(sb, images):
    sb.images = list(images)
    return sb


def test_host_parses_texture_filtering(tmp_path):
    import subprocess
    subprocess.check_call(["make", "-s", "-C", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "nano-kazen_b200", "host")])
    (tmp_path / "q.obj").write_text("v -1 -1 0\nv 1 -1 0\nv 1 1 0\nv -1 1 0\nf 1 2 3 4\n")
    mesh = "<camera type='perspective'/><mesh type='obj'><string name='filename' value='q.obj'/><bsdf type='diffuse'/></mesh></scene>"
    for integ, want in (("<integrator type='path_mis'><boolean name='textureFiltering' value='true'/></integrator>", 1),
                        ("<integrator type='path_mis'/>", 0), ("<integrator type='whitted'/>", 0)):
        (tmp_path / "s.xml").write_text("<scene>" + integ + mesh)
        hs = pk.HostScene(str(tmp_path / "s.xml"))
        assert hs.desc.integrator.texture_filtering == want
        assert f"textureFiltering={want}," in hs.describe()
        hs.close()


# ------------------------------------------------------------------------------------------------ GPU
def _gpu_count():
    import torch
    return torch.cuda.device_count()


def gpu(sb, **kw):
    g = pk.Gpu(sb.desc(), **kw)
    g.builder = sb
    return g


def _rays_into(sb, n, seed, origin):
    """rays from `origin` towards random points of the scene's box"""
    rng = np.random.default_rng(seed)
    tgt = rng.uniform(-1, 1, (n, 3))
    d = tgt - np.asarray(origin)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    r = np.zeros(n, pk.RAY_DTYPE)
    r["o"] = origin; r["d"] = d; r["tmin"] = 1e-4; r["tmax"] = 1e30
    return r


@pytest.mark.gpu
def test_probes_match_host_emulation(gpu_lib, tf):
    for thin in (None, (0.05, 3.4)):
        sb = scenes.cornell_scene(96, 64, 4, "independent", with_texture=True, normalmap=True, thinlens=thin)
        sb.set_integrator(texture_filtering=True)
        G, E = gpu(sb), tf.FootprintEmu(sb.desc())
        for origin in ((0, 0, -3.4), (0.3, -0.5, 0.2)):
            rays = _rays_into(sb, 100000, 11, origin)
            g, h = G.texture_footprint_dump(rays), E.texture_footprint_dump(rays)
            assert (g[:, 0] == h[:, 0]).all()
            hit = g[:, 0] >= 0
            assert hit.mean() > 0.9
            np.testing.assert_allclose(g[hit, 1:3], h[hit, 1:3], rtol=1e-5, atol=1e-6)
            scale = np.maximum(np.linalg.norm(h[hit, 3:7], axis=1, keepdims=True), 1e-30)
            err = np.abs(g[hit, 3:7] - h[hit, 3:7]) / scale
            # float contraction differs between nvcc and g++; grazing hits amplify it, so a small share may differ more
            assert (err.max(1) <= 1e-5).mean() >= 0.999 and err.max() <= 1e-2, err.max()
        E.close()
        # the filtered lookup over the resident pyramid vs the emulation over the numpy box pyramid of the same image
        for i, im in enumerate(sb.images):
            img = np.ctypeslib.as_array(im.rgb, shape=(im.height, im.width, 3)).copy()
            levels = box_pyramid(img)
            rng = np.random.default_rng(40 + i)
            st = rng.uniform(-1, 2, (100000, 2)).astype(np.float32)
            dst = (rng.normal(size=(100000, 4)) * 10.0 ** rng.uniform(-4, 0.5, (100000, 1))).astype(np.float32)
            np.testing.assert_allclose(G.image_lookup_filtered(i, st, dst), tf.lookup_filtered(levels, st, dst), rtol=1e-5, atol=1e-6)
            # the resident pyramid is the one kzgpu_image_lookup builds without texture filtering
            off = scenes.cornell_scene(96, 64, 4, "independent", with_texture=True, normalmap=True, thinlens=thin)
            Goff = gpu(off)
            for level in range(len(levels) + 1):
                assert G.image_lookup(i, st[:4096], level).tobytes() == Goff.image_lookup(i, st[:4096], level).tobytes(), level
            Goff.close()
        G.close()
    G = gpu(scenes.cornell_scene(32, 32, 1, with_texture=True))
    with pytest.raises(RuntimeError, match="image_lookup_filtered failed \\(-4\\)"):
        G.image_lookup_filtered(0, np.zeros((1, 2)), np.zeros((1, 4)))
    G.close()


def _frame_and_counters(sb):
    G = gpu(sb)
    f = G.render()
    s = G.stats()
    G.close()
    return f, (s["paths"], s["rays_extension"], s["rays_shadow"], s["vertices"], s["kernel_launches"])


def _quad_scene(img, filtering, spp=64, width=64, scale=1.0, background=None, kiss=True, light=True, sampler="independent", seed=1):
    """a fronto-parallel textured quad filling the frame of a 45 degree camera at distance 2, optionally lit by an emitter behind the camera"""
    sb = pk.SceneBuilder()
    h = 2.0 * math.tan(math.radians(22.5)) * 2.0
    P = np.array([[-h / 2, -h / 2, 0], [h / 2, -h / 2, 0], [h / 2, h / 2, 0], [-h / 2, h / 2, 0]], np.float32) * 1.02
    F = np.array([[0, 1, 2], [0, 2, 3]], np.uint32)
    UV = np.array([[1, 0], [0, 0], [0, 1], [1, 1]], np.float32)
    tex = sb.tex_image(img, scale=scale, srgb=False)
    const = sb.tex_constant((0.3, 0.3, 0.3))
    b = sb.bsdf_kiss(tex, const, sb.tex_constant((0, 0, 0))) if kiss else sb.bsdf_lambertian(tex)
    sb.mesh(P, F, b, normals=np.tile([[0, 0, -1]], (4, 1)), uvs=UV)
    if light:
        L = np.array([[-1, -1, -3], [1, -1, -3], [1, 1, -3], [-1, 1, -3]], np.float32)
        sb.mesh(L, np.array([[0, 2, 1], [0, 3, 2]], np.uint32), sb.bsdf_diffuse(), light=sb.light((4, 4, 4)))
    if background is not None:
        sb.background = background(sb)
    sb.set_camera(width, width, 45.0, pk.lookat((0, 0, -2), (0, 0, 0), (0, 1, 0)), near=0.1, far=100.0)
    sb.set_sampler(sampler, spp, seed=seed)
    sb.set_integrator(texture_filtering=filtering)
    return sb


NO_COUNT = {
    "constants_only": lambda on: scenes.cornell_scene(48, 48, 16, "independent", background=(0.1, 0.2, 0.3)),
    "image_background_only": lambda on: scenes.cornell_scene(48, 48, 16, "independent"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(NO_COUNT))
def test_no_counted_image_changes_nothing(gpu_lib, case):
    runs = []
    for on in (False, True):
        sb = NO_COUNT[case](on)
        if case == "image_background_only":
            img = np.random.default_rng(2).uniform(0, 1, (32, 64, 3)).astype(np.float32)
            sb.background = sb.tex_background(1.0, sb.tex_image(img, srgb=False))
        sb.set_integrator(texture_filtering=on)
        runs.append(_frame_and_counters(sb))
    # the frame sums splats with atomics in no fixed order, so two renders of one build agree to float rounding (test_multi_device_context's
    # tolerance); the counters, launches included, are exact
    np.testing.assert_allclose(runs[1][0], runs[0][0], rtol=1e-4, atol=1e-5)
    assert runs[0][1] == runs[1][1]


@pytest.mark.gpu
def test_magnified_texture_is_the_reference(gpu_lib):
    """an 8x8 texture over a 64x64 frame: lambda = log2(2 * 8 / 64 * 1.something) < 0 at every point of the quad, which is the only
    textured surface, so every lookup is the level-0 one"""
    img = np.random.default_rng(4).uniform(0, 1, (8, 8, 3)).astype(np.float32)
    frames, counters = [], []
    for on in (False, True):
        sb = _quad_scene(img, on, spp=64)
        G = gpu(sb)
        frames.append(G.render())
        s = G.stats()
        counters.append((s["paths"], s["rays_extension"], s["rays_shadow"], s["vertices"]))
        if on:
            r = _rays_into(sb, 20000, 3, (0, 0, -2))
            fp = G.texture_footprint_dump(r)
            hit = fp[:, 0] == 0
            lam = np.log2(2 * np.max(np.abs(fp[hit, 3:7]) * 8, axis=1))
            assert hit.mean() > 0.5 and lam.max() < 0
        G.close()
    np.testing.assert_allclose(frames[1], frames[0], rtol=1e-4, atol=1e-5)      # atomics: float rounding, see above
    assert counters[0] == counters[1]


def _checker(n=1024):
    y, x = np.mgrid[0:n, 0:n]
    c = ((x + y) % 2).astype(np.float32)
    return np.repeat(c[:, :, None], 3, 2)


@pytest.mark.gpu
def test_minified_checker_converges(gpu_lib):
    """1024^2 one-texel checker on a quad filling a 128^2 frame, lit by a constant environment (lambertian: every path's estimate is
    the texel it reads): at 1 spp filtering leaves a tenth of the flag-off error, and keeps the mean"""
    img = _checker()
    bg = lambda sb: sb.tex_background(1.0, sb.tex_constant((1, 1, 1)))
    mk = lambda on, spp, seed: _quad_scene(img, on, spp=spp, width=128, kiss=False, light=False, background=bg, seed=seed)
    ref_sb = mk(False, 4096, 99)
    Gr = gpu(ref_sb)
    _, _, b = Gr.frame_shape()
    ref = Gr.resolve(Gr.render())[0]
    Gr.close()
    rel = lambda a: float((((a - ref) ** 2) / (ref ** 2 + 1e-2)).mean())
    errs = {False: [], True: []}
    means = []
    for seed in range(16):
        for on in (False, True):
            G = gpu(mk(on, 1, seed))
            x = G.resolve(G.render())[0]
            G.close()
            errs[on].append(rel(x))
            if on:
                means.append(x.mean())
    off, on = np.mean(errs[False]), np.mean(errs[True])
    assert on <= 0.1 * off, (on, off)
    assert abs(np.mean(means) / ref.mean() - 1) <= 0.01, (np.mean(means), ref.mean())


@pytest.mark.gpu
def test_footprint_follows_camera_update(gpu_lib):
    img = np.random.default_rng(6).uniform(0, 1, (64, 64, 3)).astype(np.float32)
    sb = _quad_scene(img, True)
    G = gpu(sb)
    # points on the optical axis: the footprint's orientation (pbrt's RotateFromTo frame) depends on the direction from the camera, so only
    # there does moving the camera back scale it and nothing else
    r = np.zeros(64, pk.RAY_DTYPE)
    r["o"] = (0, 0, -2); r["tmin"] = 1e-4; r["tmax"] = 1e30
    r["d"] = np.stack([np.linspace(-1e-6, 1e-6, 64), np.zeros(64), np.ones(64)], -1)
    a = G.texture_footprint_dump(r)
    G.camera_update(64, 64, 45.0, pk.lookat((0, 0, -4), (0, 0, 0), (0, 1, 0)), near=0.1, far=100.0)
    b = G.texture_footprint_dump(r)
    G.close()
    hit = a[:, 0] == 0
    assert hit.all()
    n = np.linalg.norm(a[:, 3:7], axis=1, keepdims=True)
    np.testing.assert_allclose(b[:, 3:7] / n, 2 * a[:, 3:7] / n, atol=1e-4)


@pytest.mark.gpu
def test_two_devices_render_like_one(gpu_lib):
    if _gpu_count() < 2:
        pytest.skip("needs two GPUs")
    sb = scenes.cornell_scene(96, 64, 64, "independent", with_texture=True)
    sb.set_integrator(texture_filtering=True)
    a = gpu(sb).render(); b = gpu(sb, devices=(0, 1)).render()
    np.testing.assert_allclose(b, a, rtol=1e-4, atol=1e-5)
