"""GPU parity: the CUDA path through the C ABI (libkzgpu.so) against the CPU oracle on identical
inputs.  Bars (BASELINE.json north_star): hit primitive/geometry IDs bit exact, hit t within 2 ulp
(here: bit exact, both sides use the same explicitly rounded Pluecker arithmetic), sampler
sequences bit exact, images within a stated relative MSE at equal spp."""
import numpy as np
import pytest

import scenes
import pykazen as pk

pytestmark = pytest.mark.gpu

IMAGE_RELMSE_TOL = 2e-4      # per channel, GPU vs oracle at EQUAL samples (same sampler sequences)


def ulp_diff(a, b):
    a = np.ascontiguousarray(a, np.float32).view(np.int32).astype(np.int64)
    b = np.ascontiguousarray(b, np.float32).view(np.int32).astype(np.int64)
    return np.abs(a - b)


def _pair(kzo, sb, builder=pk.BUILD_HOST_SAH):
    d = sb.desc()
    return kzo.Oracle(d), pk.Gpu(d, builder=builder)


@pytest.mark.parametrize("builder", [pk.BUILD_HOST_SAH, pk.BUILD_LBVH])
def test_trace_cornell(kzo, gpu_lib, builder):
    sb = scenes.cornell_scene(32, 32, 4)
    O, G = _pair(kzo, sb, builder)
    rays = np.concatenate([scenes.primary_rays(128, 39.0, (0, 0, -3.4)), scenes.incoherent_rays(100000, extent=0.95)])
    a, b = O.trace(rays, brute=True), G.trace(rays)
    assert np.array_equal(a["geom_id"], b["geom_id"]) and np.array_equal(a["prim_id"], b["prim_id"])
    assert ulp_diff(a["t"], b["t"]).max() == 0
    assert a.tobytes() == b.tobytes()
    b2 = G.trace(rays, shadow=True)
    assert b2.tobytes() == b.tobytes()
    O.close(); G.close()


@pytest.mark.parametrize("n,builder", [(1, 0), (1, 1), (2, 1), (3, 1), (4, 1), (9, 0), (9, 1), (5000, 0), (5000, 1), (200000, 0), (200000, 1)])
def test_trace_soup(kzo, gpu_lib, n, builder):
    sb = scenes.soup_scene(n)
    O, G = _pair(kzo, sb, builder)
    rays = np.concatenate([scenes.primary_rays(128), scenes.incoherent_rays(50000)])
    a, b = O.trace(rays, brute=(n <= 5000)), G.trace(rays)
    assert a.tobytes() == b.tobytes()
    st = G.stats()
    assert st["bvh_nodes"] >= 1 and st["kernel_launches"] >= 1
    O.close(); G.close()


def test_trace_edge_cases(kzo, gpu_lib):
    sb = scenes.cornell_scene(8, 8, 1)
    P = np.array([[0, 0, 0], [0.5, 0.5, 0], [1, 1, 0]], np.float32)          # zero-area triangle
    sb.mesh(P, np.array([[0, 1, 2]], np.uint32), 0)
    O, G = _pair(kzo, sb)
    assert G.trace(np.zeros(0, pk.RAY_DTYPE)).shape == (0,)
    r = np.zeros(6, pk.RAY_DTYPE)
    r["o"] = [(0, 0, -3), (0, 0, -3), (0.25, 0.25, -0.5), (0, 0, 0), (0, 0, 0), (0.3, -1, 0.1)]
    r["d"] = [(0, 0, 1), (0, 0, 1), (0, 0, 1), (1, 0, 0), (0, 1, 0), (0, 1, 0)]      # axis-aligned: zero direction components
    r["tmin"] = [1e-4, 5.0, 0.0, 0, 0, 0]
    r["tmax"] = [np.inf, 4.0, 100.0, np.inf, np.inf, np.inf]
    assert O.trace(r, brute=True).tobytes() == G.trace(r).tobytes()
    # 33, 31 and 1 rays: ragged last warp
    for n in (1, 31, 33):
        rr = scenes.incoherent_rays(n, seed=n, extent=0.9)
        assert O.trace(rr).tobytes() == G.trace(rr).tobytes()
    O.close(); G.close()


def test_occluded_walk(kzo, gpu_lib):
    sb = scenes.cornell_scene(16, 16, 4)
    O, G = _pair(kzo, sb)
    rays = scenes.incoherent_rays(100000, extent=0.97)
    rays["tmax"] *= 1.5
    (oa, sa), (ob, sb_) = O.occluded(rays, 1e-3), G.occluded(rays, 1e-3)
    assert np.array_equal(oa, ob) and np.array_equal(sa, sb_)
    assert sa.max() >= 2
    O.close(); G.close()


@pytest.mark.parametrize("kind", ["independent", "stratified", "correlated"])
def test_sampler_bit_exact(kzo, gpu_lib, kind):
    sb = scenes.cornell_scene(64, 64, 30, kind)
    O, G = _pair(kzo, sb)
    rng = np.random.default_rng(3)
    tr = np.stack([rng.integers(0, 4000, 4000), rng.integers(0, 4000, 4000), rng.integers(0, sb.sampler.sample_count, 4000)], 1).astype(np.int32)
    pat = "P2" + "1111" * 2 + "12" * 3 + "1"
    a, b = O.sample_dump(tr, pat), G.sample_dump(tr, pat)
    assert a.tobytes() == b.tobytes()
    O.close(); G.close()


def test_sampler_pmj02bn_synthetic_tables(kzo, gpu_lib):
    rng = np.random.default_rng(5)
    bn = rng.integers(0, 65536, (48, 128, 128), dtype=np.uint16)
    pm = rng.integers(0, 2 ** 32, (5, 65536, 2), dtype=np.uint32)
    sb = scenes.cornell_scene(16, 16, 16, "stratified")
    sb.set_sampler("pmj02bn", 16, tables=(bn, pm))
    O, G = _pair(kzo, sb)
    tr = np.array([[x, y, j] for x in (0, 5, 130) for y in (1, 77) for j in (0, 3, 15)], np.int32)
    assert O.sample_dump(tr, "P2121212121212").tobytes() == G.sample_dump(tr, "P2121212121212").tobytes()
    O.close(); G.close()


@pytest.mark.parametrize("thin", [None, (0.05, 3.0)])
def test_camera_rays(kzo, gpu_lib, thin):
    sb = scenes.cornell_scene(64, 48, 4, thinlens=thin)
    O, G = _pair(kzo, sb)
    rng = np.random.default_rng(2)
    s4 = rng.uniform(0, 1, (5000, 4)).astype(np.float32) * np.array([64, 48, 1, 1], np.float32)
    a, b = O.camera_rays(s4), G.camera_rays(s4)
    for k in ("o", "d", "tmin", "tmax"):
        assert np.allclose(a[k], b[k], rtol=4e-6, atol=2e-7)
    O.close(); G.close()


def test_bsdf_queries(kzo, gpu_lib):
    sb = scenes.cornell_scene(8, 8, 1, with_texture=True, normalmap=True)
    O, G = _pair(kzo, sb)
    rng = np.random.default_rng(9)
    for bsdf in range(len(sb.bsdfs)):
        if not any(m.bsdf == bsdf for m in sb.meshes):
            continue
        for _ in range(25):
            wi = rng.normal(size=3); wi[2] = abs(wi[2]) + 0.05; wi /= np.linalg.norm(wi)
            wo = rng.normal(size=3); wo[2] = abs(wo[2]) * rng.choice([1, 1, 1, -1]) + 0.01; wo /= np.linalg.norm(wo)
            uv = rng.uniform(0, 1, 2); acc = float(rng.choice([0.0, 0.3]))
            s1 = float(rng.uniform()); s2 = rng.uniform(0, 1, 2)
            for mode in (0, 1, 2):
                a = O.bsdf_query(bsdf, mode, wi, wo, uv, acc, s1, s2)
                b = G.bsdf_query(bsdf, mode, wi, wo, uv, acc, s1, s2)
                n = 3 if mode == 0 else (1 if mode == 1 else 6)
                assert np.allclose(a[:n], b[:n], rtol=5e-4, atol=2e-6), (bsdf, mode, a, b)
    O.close(); G.close()


@pytest.mark.parametrize("cfg", [
    dict(sampler="stratified"),
    dict(sampler="correlated", visible_light=True),
    dict(sampler="independent", with_texture=True, normalmap=True, regularization=True),
    dict(sampler="stratified", thinlens=(0.05, 3.2), background=(0.3, 0.4, 0.5), max_depth=3),
])
def test_render_matches_oracle(kzo, gpu_lib, cfg):
    sb = scenes.cornell_scene(96, 64, 16, **cfg)
    O, G = _pair(kzo, sb)
    fo, fg = O.render(), G.render()
    ro, so = O.resolve(fo); rg, sg = G.resolve(fg)
    assert np.allclose(fo[..., 3], fg[..., 3], rtol=1e-4, atol=1e-5)         # identical splat weights: same pixel samples
    err = scenes.rel_mse(rg, ro)
    assert err.max() < IMAGE_RELMSE_TOL, err
    assert np.abs(sg.astype(int) - so.astype(int)).mean() < 0.5
    st_o, st_g = O.stats(), G.stats()
    assert st_g["paths"] == st_o["paths"] == 96 * 64 * 16
    # the GPU skips the extension pass after the last vertex when there is no background to look up
    # (its result cannot reach the image), so it may trace fewer rays than the reference loop, never more
    assert 0.95 * st_o["rays_extension"] <= st_g["rays_extension"] <= st_o["rays_extension"] * (1 + 2e-3)
    if cfg.get("background") is not None:
        assert abs(st_g["rays_extension"] - st_o["rays_extension"]) <= 2e-3 * st_o["rays_extension"]
    assert abs(st_g["vertices"] - st_o["vertices"]) <= 2e-3 * st_o["vertices"]
    O.close(); G.close()


def test_render_small_pool_chunks(kzo, gpu_lib, monkeypatch):
    """the chunked wavefront (pool smaller than the request) == one big chunk"""
    sb = scenes.cornell_scene(50, 37, 9, "stratified")          # ragged tile edges on purpose
    d = sb.desc()
    G1 = pk.Gpu(d)
    f1 = G1.render()
    monkeypatch.setenv("KZGPU_POOL_LOG2", "12")
    G2 = pk.Gpu(d)
    f2 = G2.render()
    assert np.allclose(f1, f2, rtol=1e-4, atol=1e-5)
    O = kzo.Oracle(d)
    ro, _ = O.resolve(O.render()); rg, _ = G2.resolve(f2)
    assert scenes.rel_mse(rg, ro).max() < IMAGE_RELMSE_TOL
    G1.close(); G2.close(); O.close()


def test_render_shards_sum_to_whole(gpu_lib):
    """sample-index shards and rectangles add up to the whole frame (the multi-GPU decomposition)"""
    sb = scenes.cornell_scene(48, 48, 16, "stratified")
    G = pk.Gpu(sb.desc())
    whole = G.render()
    parts = G.render(0, 5) + G.render(5, 16)
    assert np.allclose(whole, parts, rtol=1e-4, atol=1e-5)
    tiles = G.render(rect=(0, 0, 10, 48)) + G.render(rect=(10, 0, 48, 21)) + G.render(rect=(10, 21, 48, 48))
    assert np.allclose(whole, tiles, rtol=1e-4, atol=1e-5)
    G.close()


def test_converged_image(kzo, gpu_lib):
    """north_star (2): per-channel relative MSE of a GPU render against a high-spp converged
    reference (oracle, different sampler => independent samples) is at the Monte Carlo noise level
    of the oracle's own equal-spp render."""
    ref_sb = scenes.cornell_scene(48, 48, 1024, "independent")
    O = kzo.Oracle(ref_sb.desc())
    ref, _ = O.resolve(O.render()); O.close()
    sb = scenes.cornell_scene(48, 48, 64, "stratified")
    O2, G = _pair(kzo, sb)
    rg, _ = G.resolve(G.render()); ro, _ = O2.resolve(O2.render())
    eg, eo = scenes.rel_mse(rg, ref), scenes.rel_mse(ro, ref)
    assert eg.max() < 0.05 and np.all(eg < 1.25 * eo + 1e-4), (eg, eo)
    O2.close(); G.close()


def test_device_resident_api(gpu_lib):
    """kzgpu_trace_device / kzgpu_render_device on torch-owned HBM buffers and torch's stream"""
    import torch
    sb = scenes.soup_scene(20000)
    G = pk.Gpu(sb.desc(), builder=pk.BUILD_LBVH)
    rays = scenes.incoherent_rays(1 << 16)
    ref = G.trace(rays)
    d_rays = torch.from_numpy(rays.view(np.float32).reshape(-1, 8)).cuda()
    d_hits = torch.empty((rays.shape[0], 5), dtype=torch.float32, device="cuda")
    G.trace_device(d_rays.data_ptr(), rays.shape[0], d_hits.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    got = d_hits.cpu().numpy().reshape(-1).view(pk.HIT_DTYPE)
    assert got.tobytes() == ref.tobytes()
    G.close()


def test_errors(gpu_lib):
    import ctypes as C
    sb = scenes.soup_scene(10)
    d = sb.desc()
    lib = C.CDLL(gpu_lib)
    lib.kzgpu_last_error.restype = C.c_char_p
    h = C.c_void_p()
    assert lib.kzgpu_create(None, 0, C.byref(h)) == 0
    rays = scenes.incoherent_rays(4); hits = np.zeros(4, pk.HIT_DTYPE)
    # trace before upload / build -> KZ_ERR_STATE
    assert lib.kzgpu_trace(h, 0, rays.ctypes.data_as(C.c_void_p), C.c_size_t(4), 0, hits.ctypes.data_as(C.c_void_p)) == -4
    assert lib.kzgpu_scene_upload(h, C.byref(d)) == 0
    assert lib.kzgpu_trace(h, 0, rays.ctypes.data_as(C.c_void_p), C.c_size_t(4), 0, hits.ctypes.data_as(C.c_void_p)) == -4
    assert lib.kzgpu_accel_build(h, 7) == -1
    assert lib.kzgpu_accel_build(h, 0) == 0
    assert lib.kzgpu_trace(h, 3, rays.ctypes.data_as(C.c_void_p), C.c_size_t(4), 0, hits.ctypes.data_as(C.c_void_p)) == -1
    bad = pk.RenderReq(0, 0, 9999, 9999, 0, 1, 1)
    frame = np.zeros((68, 68, 4), np.float32)
    assert lib.kzgpu_render(h, C.byref(bad), frame.ctypes.data_as(pk.c_float_p)) == -1
    assert b"rectangle" in lib.kzgpu_last_error(h)
    lib.kzgpu_destroy(h)


def test_mip_pyramid_resident(gpu_lib):
    """the GPU-built mip pyramid: level l is the 2x2 box filter of level l-1; the periodic B-spline lookup is a partition
    of unity, so the mean over all texel centres of a level equals that level's texel mean (== level-0 mean for 2^k sizes)"""
    sb = scenes.cornell_scene(8, 8, 1, with_texture=True)
    G = pk.Gpu(sb.desc())
    img = np.ctypeslib.as_array(sb.images[0].rgb, shape=(32, 64, 3)).copy()
    cur = img.astype(np.float64)
    for level in range(0, 6):
        h, w = cur.shape[:2]
        ys, xs = np.mgrid[0:h, 0:w]
        st = np.stack([(xs + 0.5) / w, (ys + 0.5) / h], -1).reshape(-1, 2)
        got = G.image_lookup(0, st, level).reshape(h, w, 3)
        assert np.allclose(got.mean(axis=(0, 1)), cur.mean(axis=(0, 1)), rtol=1e-4, atol=1e-5), level
        # B-spline at texel centres = (1/6, 2/3, 1/6) x (1/6, 2/3, 1/6) periodic stencil of the level's texels
        k = np.array([1 / 6, 2 / 3, 1 / 6])
        exp = sum(k[a] * k[b] * np.roll(np.roll(cur, 1 - a, axis=0), 1 - b, axis=1) for a in range(3) for b in range(3))
        assert np.allclose(got, exp, rtol=1e-4, atol=1e-5), level
        if h == 1 and w == 1:
            break
        nh, nw = max(1, h // 2), max(1, w // 2)
        cur = 0.25 * (cur[0:2 * nh:2, 0:2 * nw:2] + cur[0:2 * nh:2, 1:2 * nw:2] + cur[1:2 * nh:2, 0:2 * nw:2] + cur[1:2 * nh:2, 1:2 * nw:2]) if h > 1 and w > 1 else cur
    G.close()


def test_extra_bsdf_queries_gpu(kzo, gpu_lib):
    sb = scenes.gallery_scene(8, 8, 1)
    O, G = _pair(kzo, sb)
    rng = np.random.default_rng(13)
    for bsdf in range(len(sb.bsdfs)):
        if not any(m.bsdf == bsdf for m in sb.meshes):
            continue
        for _ in range(25):
            wi = rng.normal(size=3); wi[2] = (abs(wi[2]) + 0.05) * rng.choice([1, 1, 1, -1]); wi /= np.linalg.norm(wi)
            wo = rng.normal(size=3); wo[2] = (abs(wo[2]) + 0.02) * rng.choice([1, 1, -1]); wo /= np.linalg.norm(wo)
            uv = rng.uniform(0, 1, 2); s1 = float(rng.uniform()); s2 = rng.uniform(0.001, 0.999, 2)
            for mode in (0, 1, 2):
                a = O.bsdf_query(bsdf, mode, wi, wo, uv, 0.0, s1, s2)
                b = G.bsdf_query(bsdf, mode, wi, wo, uv, 0.0, s1, s2)
                n = 3 if mode == 0 else (1 if mode == 1 else 7)
                assert np.allclose(a[:n], b[:n], rtol=2e-3, atol=5e-6), (sb.bsdfs[bsdf].type, mode, a, b)
    O.close(); G.close()


def test_extra_bsdf_render_gpu(kzo, gpu_lib):
    """refraction (eta), discrete measures (bsdfWeight = 1), Beckmann lobes and the generic material class on the GPU"""
    sb = scenes.gallery_scene(96, 72, 16)
    O, G = _pair(kzo, sb)
    ro, _ = O.resolve(O.render()); rg, _ = G.resolve(G.render())
    err = scenes.rel_mse(rg, ro)
    assert err.max() < 1e-3, err            # specular chains amplify libm-level differences; still far below MC noise
    st_o, st_g = O.stats(), G.stats()
    assert abs(st_g["vertices"] - st_o["vertices"]) <= 5e-3 * st_o["vertices"]
    O.close(); G.close()


@pytest.mark.parametrize("kind", ["normals", "ao", "whitted", "path_mats"])
def test_other_integrators_gpu(kzo, gpu_lib, kind):
    sb = scenes.cornell_scene(64, 48, 16, "stratified", visible_light=True)
    sb.set_integrator(kind=kind)
    O, G = _pair(kzo, sb)
    ro, _ = O.resolve(O.render()); rg, _ = G.resolve(G.render())
    # whitted is ill-conditioned by construction (see tests/test_hostemu.py): statistical tolerance
    assert scenes.rel_mse(rg, ro).max() < (1e-6 if kind == "normals" else (2e-2 if kind == "whitted" else 5e-4))
    assert G.stats()["paths"] == 64 * 48 * 16
    O.close(); G.close()


def _tie_scene():
    """two meshes holding the SAME triangle (exact t tie) + a coplanar shifted copy: the documented tie rule is
    smallest (geomID, primID) -- independent of BVH and traversal order (SURVEY Appendix C)"""
    sb = pk.SceneBuilder()
    m = sb.bsdf_diffuse((0.5, 0.5, 0.5))
    T = np.array([[-1, -1, 0.5], [1, -1, 0.5], [0, 1, 0.5]], np.float32)
    F = np.array([[0, 1, 2]], np.uint32)
    sb.mesh(np.concatenate([T + np.float32([0.25, 0, 0]), T]), np.array([[0, 1, 2], [3, 4, 5]], np.uint32), m)      # geom 0: prim 1 == the shared triangle
    sb.mesh(T, F, m)                                                                                               # geom 1: prim 0 == the shared triangle
    sb.mesh(np.concatenate([T, T]), np.array([[3, 4, 5], [0, 1, 2]], np.uint32), m)                                # geom 2: twice
    sb.set_camera(16, 16, 40.0, pk.lookat((0, 0, -3), (0, 0, 0), (0, 1, 0)))
    return sb


@pytest.mark.parametrize("builder", [pk.BUILD_HOST_SAH, pk.BUILD_LBVH])
def test_exact_ties_resolve_by_ids(kzo, gpu_lib, builder):
    sb = _tie_scene()
    O, G = _pair(kzo, sb, builder)
    rays = scenes.primary_rays(96, 40.0, (0, 0, -3.0))
    a, b = O.trace(rays, brute=True), G.trace(rays)
    assert a.tobytes() == b.tobytes() == O.trace(rays, brute=False).tobytes()
    hit = a["geom_id"] != 0xFFFFFFFF
    assert hit.any() and (a["geom_id"][hit] == 0).all()              # geom 0 always wins a tie
    # where only the shared triangle is hit (outside the shifted copy) prim 1 of geom 0 is reported; in the overlap prim 0 < prim 1 wins
    assert set(np.unique(a["prim_id"][hit]).tolist()) == {0, 1}
    O.close(); G.close()


def test_empty_and_tiny_scenes(kzo, gpu_lib):
    """no meshes at all (empty accel), a single triangle, a 1x1 film, one sample"""
    sb = pk.SceneBuilder()
    sb.set_camera(1, 1, 40.0, pk.lookat((0, 0, -3), (0, 0, 0), (0, 1, 0)))
    sb.set_sampler("stratified", 1)
    sb.background = sb.tex_background(2.0, sb.tex_constant((0.1, 0.2, 0.3)))
    for builder in (pk.BUILD_HOST_SAH, pk.BUILD_LBVH):
        G = pk.Gpu(sb.desc(), builder=builder)
        rays = scenes.incoherent_rays(100)
        h = G.trace(rays)
        assert (h["geom_id"] == 0xFFFFFFFF).all() and np.array_equal(h["t"], rays["tmax"])
        f = G.render()
        rgb, _ = G.resolve(f)
        assert rgb.shape == (1, 1, 3) and np.all(rgb == 0)             # camera rays never see the background (integrator.cpp:210-212)
        occ, seg = G.occluded(rays, 1e-3)
        assert not occ.any() and (seg == 1).all()
        G.close()
    sb.mesh(np.array([[-5, -5, 1], [5, -5, 1], [0, 5, 1]], np.float32), np.array([[0, 2, 1]], np.uint32), sb.bsdf_diffuse((0.5, 0.5, 0.5)))
    O, G = _pair(kzo, sb)
    fo, fg = O.render(), G.render()
    assert np.allclose(fo, fg, rtol=1e-5, atol=1e-6) and fo[..., :3].max() > 0          # one bounce to the background
    O.close(); G.close()


def test_far_from_origin_and_huge_triangles(kzo, gpu_lib):
    """coordinates around 1e4 with millimetre triangles next to kilometre ones: culling stays conservative"""
    rng = np.random.default_rng(4)
    n = 3000
    c = rng.uniform(-1, 1, (n, 1, 3)).astype(np.float32) * np.float32(50) + np.float32(1e4)
    P = (c + rng.uniform(-0.5, 0.5, (n, 3, 3)).astype(np.float32)).reshape(-1, 3)
    big = np.array([[9000, 9000, 10060], [11000, 9000, 10060], [10000, 11000, 10060]], np.float32)
    P = np.concatenate([P, big])
    F = np.arange(P.shape[0], dtype=np.uint32).reshape(-1, 3)
    sb = pk.SceneBuilder()
    sb.mesh(P, F, sb.bsdf_diffuse((0.5, 0.5, 0.5)))
    sb.set_camera(8, 8, 40.0, pk.lookat((1e4, 1e4, 1e4 - 200), (1e4, 1e4, 1e4), (0, 1, 0)))
    rays = scenes.incoherent_rays(20000, extent=60.0)
    rays["o"] += np.float32(1e4); rays["tmax"] = 500.0
    for builder in (pk.BUILD_HOST_SAH, pk.BUILD_LBVH):
        O, G = _pair(kzo, sb, builder)
        a, b = O.trace(rays, brute=True), G.trace(rays)
        assert a.tobytes() == b.tobytes() and (a["geom_id"] != 0xFFFFFFFF).mean() > 0.3
        O.close(); G.close()


def test_render_rect_and_spp_edges(kzo, gpu_lib):
    """non-square sample counts, a one-pixel-wide rectangle, maxDepth 1, tent and box filters (border 1 and 0)"""
    for filt in ("tent", "box", "mitchell"):
        sb = scenes.cornell_scene(33, 17, 7, "correlated", max_depth=1)
        sb.set_filter(filt)
        O, G = _pair(kzo, sb)
        fo, fg = O.render(), G.render()
        ro, _ = O.resolve(fo); rg, _ = G.resolve(fg)
        assert fo.shape == fg.shape and scenes.rel_mse(rg, ro).max() < IMAGE_RELMSE_TOL
        part_o = O.render(2, 5, rect=(16, 3, 17, 11)); part_g = G.render(2, 5, rect=(16, 3, 17, 11))
        assert np.allclose(part_o, part_g, rtol=1e-3, atol=1e-5)
        O.close(); G.close()


def test_multi_device_context(kzo, gpu_lib):
    """one kzgpu_ctx over all visible devices: sample-index shards rendered concurrently, frames summed (SURVEY 8e)"""
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    sb = scenes.cornell_scene(64, 64, 16, "stratified", with_texture=True)
    d = sb.desc()
    rays = scenes.incoherent_rays(10000, extent=0.9)
    for builder in (pk.BUILD_HOST_SAH, pk.BUILD_LBVH):           # LBVH: built on device 0, replicated over NVLink
        G1 = pk.Gpu(d, devices=(0,), builder=builder)
        GN = pk.Gpu(d, devices=tuple(range(n)), builder=builder)
        f1, fn = G1.render(), GN.render()
        assert np.allclose(f1, fn, rtol=1e-4, atol=1e-5)
        st = GN.stats()
        assert st["paths"] == 64 * 64 * 16 and st["ms_merge"] > 0          # the frames were merged on the devices (k_frame_reduce)
        assert G1.trace(rays).tobytes() == GN.trace(rays, device=n - 1).tobytes()
        # progressive: a second request adds to the frame passed in (clear_frame = 0), on one device as on N
        half = GN.render(0, 8)
        full = GN.render(8, 16, frame=half.copy())
        assert np.allclose(full, fn, rtol=1e-4, atol=1e-5)
        G1.close(); GN.close()


def test_nan_rays_are_misses(kzo, gpu_lib):
    """NaN rays (the cosine-hemisphere warp yields one for a sample that is exactly 0) are immediate misses, not full-tree walks"""
    import time
    sb = scenes.soup_scene(200000)
    O, G = _pair(kzo, sb, pk.BUILD_LBVH)
    rays = scenes.incoherent_rays(4096)
    rays["d"][::7, 0] = np.nan; rays["o"][3::11, 2] = np.nan; rays["tmax"][5::13] = np.nan
    t0 = time.time(); b = G.trace(rays); dt = time.time() - t0
    a = O.trace(rays)
    assert a.tobytes() == b.tobytes()
    bad = np.isnan(rays["d"]).any(1) | np.isnan(rays["o"]).any(1) | np.isnan(rays["tmax"])
    assert (b["geom_id"][bad] == 0xFFFFFFFF).all() and dt < 2.0
    O.close(); G.close()


def test_studio_scene_matches_oracle(kzo, gpu_lib):
    """the WarmStudio stand-in (BASELINE configs[0] class): smooth 15 872-triangle kiss ball, invisible light array, mitchell filter"""
    sb = scenes.studio_scene(160, 90, 16)
    O, G = _pair(kzo, sb)
    ro, _ = O.resolve(O.render()); rg, _ = G.resolve(G.render())
    assert scenes.rel_mse(rg, ro).max() < IMAGE_RELMSE_TOL
    assert 0.005 < ro.mean() < 0.2
    O.close(); G.close()


def test_c4_standin_pmj02bn_terminator_regularization(kzo, gpu_lib):
    """BASELINE configs[3] stand-in: pmj02bn sampler (stand-in tables from the C++ host: the pbrt tables are not in the reference's
    public tree), low-poly smooth-shaded sphere (Hanika shadow-terminator offset, accel.cpp:141-153), per-bounce roughness bias"""
    bn, pm = pk.host_fallback_tables()
    sb = scenes.cornell_scene(96, 54, 16, "stratified", regularization=True, with_texture=True)
    P, N, UV, F = scenes.uv_sphere((0.45, 0.1, -0.2), 0.3, nu=8, nv=5)          # coarse: terminator artefacts without the offset
    sb.mesh(P, F, sb.bsdf_kiss(sb.tex_constant((0.8, 0.8, 0.8)), sb.tex_constant((0.3, 0, 0)), sb.tex_constant((0.0, 0, 0))), normals=N, uvs=UV)
    sb.set_sampler("pmj02bn", 16, tables=(bn, pm))
    sb.set_integrator(max_depth=6, regularization=True, accumulated_roughness=0.5)
    O, G = _pair(kzo, sb)
    tr = np.array([[x, y, j] for x in (0, 17, 95) for y in (2, 53) for j in (0, 7, 15)], np.int32)
    assert O.sample_dump(tr, "P2121212121212").tobytes() == G.sample_dump(tr, "P2121212121212").tobytes()
    ro, _ = O.resolve(O.render()); rg, _ = G.resolve(G.render())
    assert scenes.rel_mse(rg, ro).max() < IMAGE_RELMSE_TOL
    O.close(); G.close()


def test_latlong_environment_map(kzo, gpu_lib):
    """image-backed background (BackgroundTexture -> ImageTexture::eval(dir), texture.cpp:66-81,121-126): lat-long lookup on the GPU"""
    rng = np.random.default_rng(17)
    env = rng.uniform(0.0, 2.0, (16, 32, 3)).astype(np.float32)
    sb = scenes.cornell_scene(64, 48, 16, "stratified", max_depth=4)
    sb.background = sb.tex_background(1.5, sb.tex_image(env, srgb=False))
    # open the box: drop the ceiling and the light meshes so that most paths escape to the environment
    sb.meshes = [m for i, m in enumerate(sb.meshes) if i != 1 and m.light < 0]
    O, G = _pair(kzo, sb)
    ro, _ = O.resolve(O.render()); rg, _ = G.resolve(G.render())
    assert ro.mean() > 0.05 and scenes.rel_mse(rg, ro).max() < IMAGE_RELMSE_TOL
    O.close(); G.close()


@pytest.mark.parametrize("n_tris", [1 << 20, 10_000_000])
def test_full_size_properties(gpu_lib, n_tris):
    """BASELINE configs[1] sizes (1 M and 10 M triangle soup, 2^22-ray batches): size-independent properties instead of the
    oracle, which would need minutes here.
      - the hit does not depend on the accel: GPU-built LBVH and host SAH return identical bytes (1 M only: the host SAH of 10 M
        triangles takes too long for a test);
      - clipping: re-tracing a hit ray with tmax = t returns the same hit (the interval is closed), with tmax just below t a miss
        (t was the closest hit) -- the erase/decode round trip of this domain;
      - batching: a permuted batch returns the permuted hits, two half batches return the whole;
      - occlusion: with no invisible lights the occlusion walk is `hit exists` with one segment per ray."""
    sb = scenes.soup_scene(n_tris)
    d = sb.desc()
    G = pk.Gpu(d, builder=pk.BUILD_LBVH)
    rays = np.concatenate([scenes.primary_rays(1024), scenes.incoherent_rays((1 << 22) - (1 << 20))])
    h = G.trace(rays)
    hit = h["geom_id"] != 0xFFFFFFFF
    assert 0.5 < hit.mean() < 1.0
    assert np.all(h["t"][hit] >= rays["tmin"][hit]) and np.all(h["t"][hit] <= rays["tmax"][hit])
    assert np.all(h["prim_id"][hit] < n_tris) and np.all(h["geom_id"][hit] == 0)
    if n_tris <= (1 << 20):
        G2 = pk.Gpu(d, builder=pk.BUILD_HOST_SAH)
        assert G2.trace(rays).tobytes() == h.tobytes()
        G2.close()
    # clipping round trip
    clip = rays[hit].copy(); clip["tmax"] = h["t"][hit]
    hc = G.trace(clip)
    assert hc.tobytes() == h[hit].tobytes()
    clip["tmax"] = np.nextafter(h["t"][hit], np.float32(0))
    below = G.trace(clip)
    assert np.all(below["geom_id"] == 0xFFFFFFFF)
    # batching
    perm = np.random.default_rng(3).permutation(len(rays))
    assert G.trace(rays[perm]).tobytes() == h[perm].tobytes()
    half = len(rays) // 2
    assert np.concatenate([G.trace(rays[:half]), G.trace(rays[half:])]).tobytes() == h.tobytes()
    # occlusion walk without invisible lights
    occ, seg = G.occluded(rays[: 1 << 20], 1e-4)
    assert np.array_equal(occ.astype(bool), hit[: 1 << 20]) and np.all(seg == 1)
    G.close()


@pytest.mark.parametrize("n_tris", [1 << 20, 10_000_000])
def test_full_size_sampled_oracle(kzo, gpu_lib, n_tris):
    """BASELINE configs[1] at full size against the oracle: the GPU-built LBVH accel of the 1 M / 10 M triangle soup and the
    oracle's BVH2 over the same triangles return identical bytes for 2^18 primary + 2^18 incoherent rays (a sample of the
    bench batches: same generators, same seeds)."""
    sb = scenes.soup_scene(n_tris)
    d = sb.desc()
    G = pk.Gpu(d, builder=pk.BUILD_LBVH)
    O = kzo.Oracle(d)
    rays = np.concatenate([scenes.primary_rays(512), scenes.incoherent_rays(1 << 18)])
    a, b = O.trace(rays), G.trace(rays)
    assert a.tobytes() == b.tobytes()
    assert 0.5 < (a["geom_id"] != 0xFFFFFFFF).mean() < 1.0
    occ_o, seg_o = O.occluded(rays[-(1 << 16):], 1e-4)
    occ_g, seg_g = G.occluded(rays[-(1 << 16):], 1e-4)
    assert np.array_equal(occ_o, occ_g) and np.array_equal(seg_o, seg_g)
    O.close(); G.close()


def test_intersection_record(kzo, gpu_lib):
    """A3 on the device, field by field (accel.cpp:113-236): all three shading-frame cases, textured and untextured meshes."""
    from test_hostemu import check_intersection_dump
    for sb, rays in ((scenes.cornell_scene(16, 16, 4, with_texture=True, normalmap=True),
                      np.concatenate([scenes.primary_rays(96, 39.0, (0, 0, -3.4)), scenes.incoherent_rays(40000, extent=0.95)])),
                     (scenes.gallery_scene(16, 12, 4),
                      np.concatenate([scenes.primary_rays(96, 50.0, (0, 0.1, -3.2)), scenes.incoherent_rays(40000, extent=0.9)]))):
        for builder in (pk.BUILD_HOST_SAH, pk.BUILD_LBVH):
            O, G = _pair(kzo, sb, builder)
            check_intersection_dump(O, G, rays)
            O.close(); G.close()


def test_emitter_sample(kzo, gpu_lib):
    """S1 / L1 / L2 on the device, field by field (scene.h:45-56, mesh.cpp:108-133, light.cpp:16-51)."""
    from test_hostemu import check_light_sample_dump
    O, G = _pair(kzo, scenes.cornell_scene(16, 16, 4))
    check_light_sample_dump(O, G, n=50000)
    O.close(); G.close()
    sb = scenes.studio_scene(16, 16, 4)                    # one emitter of 32 triangles: exercises the area CDF
    O, G = _pair(kzo, sb)
    rng = np.random.default_rng(9)
    ref = rng.uniform(-1.0, 1.0, (20000, 3)).astype(np.float32) + np.array([0, 1, 0], np.float32)
    u5 = rng.uniform(0, 1, (20000, 5)).astype(np.float32)
    a, b = O.light_sample_dump(ref, u5), G.light_sample_dump(ref, u5)
    assert a[:, 0].tobytes() == b[:, 0].tobytes()
    np.testing.assert_allclose(b[:, 1:11], a[:, 1:11], rtol=2e-5, atol=2e-6)
    O.close(); G.close()


def test_scene_ingest_from_device_arrays(kzo, gpu_lib):
    """kz_mesh_desc arrays may be CUDA device pointers (read in place by the ingest kernels): same accel, same hits, same image
    as the host-array upload -- including an emitter, whose arrays are read back for the area CDF."""
    import ctypes as C
    torch = pytest.importorskip("torch")
    sb = scenes.cornell_scene(48, 48, 16, with_texture=True)
    d = sb.desc()
    keep = []
    dd = pk.SceneDesc.from_buffer_copy(d)
    meshes = (pk.MeshDesc * d.n_meshes)()
    for g in range(d.n_meshes):
        m = d.meshes[g]
        C.memmove(C.byref(meshes[g]), C.byref(m), C.sizeof(pk.MeshDesc))
        for name, per, cnt, ctype in (("positions", 3, m.n_vertices, C.c_float), ("normals", 3, m.n_vertices, C.c_float),
                                      ("uvs", 2, m.n_vertices, C.c_float), ("indices", 3, m.n_triangles, C.c_uint32)):
            src = getattr(m, name)
            if not src:
                continue
            host = np.ctypeslib.as_array(src, shape=(cnt * per,)).copy()
            t = torch.from_numpy(host.view(np.float32 if ctype is C.c_float else np.int32)).cuda()
            keep.append(t)
            setattr(meshes[g], name, C.cast(t.data_ptr(), C.POINTER(ctype)))
    dd.meshes = meshes
    rays = np.concatenate([scenes.primary_rays(96, 39.0, (0, 0, -3.4)), scenes.incoherent_rays(30000, extent=0.95)])
    for builder in (pk.BUILD_HOST_SAH, pk.BUILD_LBVH):
        G1, G2 = pk.Gpu(d, builder=builder), pk.Gpu(dd, builder=builder)
        assert G1.trace(rays).tobytes() == G2.trace(rays).tobytes()
        assert G1.render().tobytes() == G2.render().tobytes() or scenes.rel_mse(G2.resolve(G2.render())[0], G1.resolve(G1.render())[0]).max() < 1e-9
        G1.close(); G2.close()


def test_upload_validation(gpu_lib):
    """kzgpu_scene_upload rejects what the device code cannot hold instead of reading out of bounds."""
    sb = scenes.cornell_scene(8, 8, 1)
    P = np.zeros((3, 3), np.float32)
    sb.mesh(P, np.array([[0, 1, 3]], np.uint32), 0)                       # vertex index out of range (checked on the device)
    with pytest.raises(RuntimeError, match="vertex index out of range"):
        pk.Gpu(sb.desc())
    sb = scenes.cornell_scene(8, 8, 1)
    sb.mesh(np.zeros((3, 3), np.float32), np.zeros((0, 3), np.uint32), 0, light=sb.light((1, 1, 1)))
    with pytest.raises(RuntimeError, match="emissive mesh without triangles"):
        pk.Gpu(sb.desc())
    sb = scenes.cornell_scene(8, 8, 1)
    t = sb.tex_constant((1, 1, 1))
    for _ in range(5):
        t = sb.tex_colorramp(0.0, 1.0, t)                                    # six levels deep
    sb.mesh(*scenes.quad((0, 0, 0), (1, 0, 0), (1, 1, 0), (0, 1, 0)), sb.bsdf_lambertian(t))
    with pytest.raises(RuntimeError, match="deeper than"):
        pk.Gpu(sb.desc())
    sb = scenes.cornell_scene(8, 8, 1)
    a = sb.tex_colorramp(0.0, 1.0, 0); b = sb.tex_colorramp(0.0, 1.0, a); sb.textures[a].child[0] = b      # cycle
    with pytest.raises(RuntimeError, match="cycle"):
        pk.Gpu(sb.desc())
    bn, pm = pk.host_fallback_tables()
    sb = scenes.cornell_scene(8, 8, 4)
    sb.set_sampler("pmj02bn", 4, tables=(bn, pm))
    G = pk.Gpu(sb.desc())
    with pytest.raises(RuntimeError, match="sample_count"):
        G.render(0, 5)                                                       # pmj02bn tables hold sample_count entries per pixel
    G.render(0, 4)
    G.close()


def test_lanes_and_pool_sizes_agree(gpu_lib, monkeypatch):
    """One lane, two lanes, four lanes, small pools and every path order (runs of 1 / 5 / 8 / 144 sample indices per pixel tile, 5 not
    dividing the sample count) walk the same paths: identical counters, images equal up to the order of the float reductions into the frame."""
    sb = scenes.cornell_scene(160, 120, 144, "stratified")          # 2.8 M paths: enough for the lanes to engage
    d = sb.desc()
    out = []
    for lanes, pool, group in (("1", "23", "1"), ("2", "23", "8"), ("4", "19", "5"), ("2", "17", "144"), ("3", "24", "8")):
        monkeypatch.setenv("KZGPU_LANES", lanes); monkeypatch.setenv("KZGPU_POOL_LOG2", pool); monkeypatch.setenv("KZGPU_SPP_GROUP", group)
        G = pk.Gpu(d)
        f = G.render()
        rgb, _ = G.resolve(f)
        st = G.stats()
        out.append((rgb, st["paths"], st["rays_extension"], st["rays_shadow"], st["vertices"]))
        G.close()
    for o in out[1:]:
        assert o[1:] == out[0][1:]
        assert scenes.rel_mse(o[0], out[0][0]).max() < 1e-9
