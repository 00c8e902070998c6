"""Oracle pinned to the known-answer vectors generated from the reference's own hash.h / pcg32.h /
permute() (oracle/ref_kat.cpp -> tests/golden/sampler_kat.json), plus oracle self-consistency."""
import ctypes as C
import json
import os

import numpy as np
import pytest

import scenes

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def kat():
    with open(os.path.join(HERE, "golden", "sampler_kat.json")) as f:
        return json.load(f)


def test_hash16(kzo, kat):
    L = kzo.lib()
    for x, y, seed, h in kat["hash16"]:
        assert L.kzo_hash_pixel_seed(x, y, int(seed)) == int(h)


def test_hash20(kzo, kat):
    L = kzo.lib()
    for x, y, dim, seed, h in kat["hash20"]:
        assert L.kzo_hash_pixel_dim_seed(x, y, dim, int(seed)) == int(h)


def test_mixbits(kzo, kat):
    L = kzo.lib()
    for v, m in kat["mixbits"]:
        assert L.kzo_mix_bits(int(v)) == int(m)


def test_permute(kzo, kat):
    L = kzo.lib()
    for i, l, p, r in kat["permute"]:
        assert L.kzo_permute(i, l, p) == r


def test_pcg32(kzo, kat):
    L = kzo.lib()
    out = (C.c_uint32 * 3)()
    for seed, delta, a, b, fbits in kat["pcg32"]:
        L.kzo_pcg32_stream(int(seed), int(delta), out, 3)
        assert (out[0], out[1]) == (a, b)
        f = np.array([((out[2] >> 9) | 0x3F800000)], np.uint32).view(np.float32)[0] - np.float32(1.0)
        assert np.float32(f).view(np.uint32) == fbits


def test_survey_vectors(kzo, kat):
    """the six vectors quoted in SURVEY.md Appendix B"""
    L = kzo.lib()
    s = kat["survey"]
    assert int(s["hash16"]) == 0x832F7F82265C2CF0 and L.kzo_hash_pixel_seed(3, 7, 1) == 0x832F7F82265C2CF0
    assert int(s["hash20"]) == 0xB9CD4008D42A6133 and L.kzo_hash_pixel_dim_seed(3, 7, 4, 1) == 0xB9CD4008D42A6133
    assert L.kzo_mix_bits(0x832F7F82265C2CF0) == 0x5EFEE82B6FDAB425
    out = (C.c_uint32 * 1)()
    L.kzo_pcg32_stream(0x832F7F82265C2CF0, 5 * 65536, out, 1)
    assert out[0] == 0x80B3B771 == s["pcg_u"]
    assert L.kzo_permute(5, 64, 0xB9CD4008D42A6133 & 0xFFFFFFFF) == 39 == s["perm_a"]
    assert L.kzo_permute(5, 64, (0xB9CD4008D42A6133 * 0x51633E2D) & 0xFFFFFFFF) == 29 == s["perm_b"]


def test_stratified_composition(kzo):
    """next1D/next2D of the stratified sampler recomposed in numpy from the pinned primitives
    (sampler.cpp:111-156): stratum = permute(j, spp, (u32)Hash(p, dim, seed)), jitter = pcg float."""
    L = kzo.lib()
    sb = scenes.cornell_scene(16, 16, 16, "stratified")
    O = kzo.Oracle(sb.desc())
    spp, res = 16, 4
    for (px, py, j) in [(0, 0, 0), (3, 7, 5), (15, 2, 15)]:
        got = O.sample_dump(np.array([[px, py, j]], np.int32), "P1")[0]
        u = (C.c_uint32 * 3)()
        L.kzo_pcg32_stream(L.kzo_hash_pixel_seed(px, py, 1), j * 65536, u, 3)
        fl = [np.float32(np.array([(v >> 9) | 0x3F800000], np.uint32).view(np.float32)[0] - np.float32(1)) for v in u]
        s0 = L.kzo_permute(j, spp, L.kzo_hash_pixel_dim_seed(px, py, 0, 1) & 0xFFFFFFFF)
        s1 = L.kzo_permute(j, spp, L.kzo_hash_pixel_dim_seed(px, py, 2, 1) & 0xFFFFFFFF)
        exp = [np.float32(np.float32(s0 % res) + fl[0]) / np.float32(res), np.float32(np.float32(s0 // res) + fl[1]) / np.float32(res),
               np.float32(np.float32(s1) + fl[2]) / np.float32(spp)]
        assert np.array_equal(np.array(exp, np.float32).view(np.uint32), got.view(np.uint32))
    O.close()


def test_samplers_in_unit_interval_and_stratified(kzo):
    for kind in ("independent", "stratified", "correlated"):
        sb = scenes.cornell_scene(8, 8, 16, kind)
        O = kzo.Oracle(sb.desc())
        tr = np.array([[2, 3, j] for j in range(16)], np.int32)
        v = O.sample_dump(tr, "P21")
        assert (v >= 0).all() and (v < 1).all()
        if kind != "independent":
            # every one of the 16 1-D strata is hit exactly once by the 16 samples of the pixel
            assert sorted(np.floor(v[:, 4] * 16).astype(int).tolist()) == list(range(16))
            # 2-D: 4x4 strata (stratified) / 4x4 cells (cmj)
            cells = (np.floor(v[:, 0] * 4) + 4 * np.floor(v[:, 1] * 4)).astype(int)
            assert sorted(cells.tolist()) == list(range(16))
        O.close()


def test_brute_vs_bvh_hits(kzo):
    """hit identity is BVH independent: conservative BVH2 == test-every-triangle (bit exact)"""
    sb = scenes.cornell_scene(32, 32, 4)
    O = kzo.Oracle(sb.desc())
    rays = np.concatenate([scenes.primary_rays(48, 39.0, (0, 0, -3.4)), scenes.incoherent_rays(6000, extent=0.95)])
    a, b = O.trace(rays, brute=True), O.trace(rays, brute=False)
    assert a.tobytes() == b.tobytes()
    assert (a["geom_id"] != 0xFFFFFFFF).mean() > 0.5
    O.close()


def test_soup_brute_vs_bvh(kzo):
    sb = scenes.soup_scene(3000)
    O = kzo.Oracle(sb.desc())
    rays = np.concatenate([scenes.primary_rays(40), scenes.incoherent_rays(3000)])
    a, b = O.trace(rays, brute=True), O.trace(rays, brute=False)
    assert a.tobytes() == b.tobytes()
    O.close()


def test_edge_cases(kzo):
    """empty batch, degenerate triangle, ray starting on a surface, zero-length interval"""
    sb = scenes.cornell_scene(8, 8, 1)
    # a zero-area triangle must never be reported
    P = np.array([[0, 0, 0], [0.5, 0.5, 0], [1, 1, 0]], np.float32)
    sb.mesh(P, np.array([[0, 1, 2]], np.uint32), 0)
    O = kzo.Oracle(sb.desc())
    assert O.trace(np.zeros(0, scenes.pk.RAY_DTYPE)).shape == (0,)
    r = np.zeros(3, scenes.pk.RAY_DTYPE)
    r["o"] = [(0, 0, -3), (0, 0, -3), (0.25, 0.25, -0.5)]
    r["d"] = [(0, 0, 1), (0, 0, 1), (0, 0, 1)]
    r["tmin"] = [1e-4, 5.0, 0.0]
    r["tmax"] = [np.inf, 4.0, 100.0]          # second ray: empty interval
    h = O.trace(r, brute=True)
    assert h["geom_id"][0] != 0xFFFFFFFF and h["geom_id"][1] == 0xFFFFFFFF
    deg = len(sb.meshes) - 1
    assert (h["geom_id"] != deg).all()
    O.close()


def test_filter_tables(kzo):
    """pykazen's table builder (used to fill kz_filter_desc) == oracle restatement of rfilter.cpp"""
    L = kzo.lib()
    for kind, k, args in (("gaussian", 0, (2.0, 0.5, 0)), ("mitchell", 1, (2.0, 1 / 3, 1 / 3)), ("tent", 2, (0, 0, 0)), ("box", 3, (0, 0, 0))):
        rad = C.c_float(); tab = (C.c_float * 33)()
        L.kzo_filter_table(k, C.c_float(args[0]), C.c_float(args[1]), C.c_float(args[2]), C.byref(rad), tab)
        r, t = scenes.pk.filter_table(kind)
        assert abs(r - rad.value) < 1e-7
        assert np.allclose(np.array(list(tab), np.float32), t, rtol=2e-6, atol=1e-7)
        assert tab[32] == 0.0


def test_light_cdf(kzo):
    sb = scenes.cornell_scene(8, 8, 1)
    O = kzo.Oracle(sb.desc())
    lm = [i for i, m in enumerate(sb.meshes) if m.light >= 0][0]
    cdf, nrm = O.light_cdf(lm, 2)
    assert cdf[0] == 0 and cdf[-1] == 1 and abs(cdf[1] - 0.5) < 1e-6 and abs(1 / nrm - 0.36) < 1e-5
    O.close()


def test_render_converges_to_itself(kzo):
    """equal-spp renders with different sampler seeds agree within Monte Carlo noise; the frame's
    weight channel equals the sum of filter weights (no sample dropped)"""
    sb = scenes.cornell_scene(32, 32, 16, "stratified")
    O = kzo.Oracle(sb.desc())
    f = O.render()
    rgb, srgb = O.resolve(f)
    assert np.isfinite(f).all() and (f[..., 3] >= 0).all()
    assert 0.02 < rgb.mean() < 1.0
    assert srgb.dtype == np.uint8 and srgb.max() > 50
    st = O.stats()
    assert st["paths"] == 32 * 32 * 16 and st["rays_extension"] >= st["paths"]
    O.close()


def test_math_helpers_match_the_reference_bodies(kzo):
    """tests/golden/math_kat.json holds inputs and outputs of the reference's OWN function bodies (ggx_brdf.h, frame.h, dpdf.h,
    common.cpp colour helpers / fresnel / refract / reflect / coordinateSystem, warp.cpp, the eval / pdf / sample methods of
    KazenStandardSurface, Diffuse and the seven other BSDF plugins from bsdf.cpp, the background / colorramp / blend nodes of texture.cpp, and the generateSample / next1D / next2D / nextPixel2D methods of the Independent,
    Stratified and Correlated samplers from sampler.cpp) run by oracle/ref_math_kat.cpp: the oracle's restatements must reproduce every
    output bit for bit."""
    import json
    g = json.load(open(os.path.join(HERE, "golden", "math_kat.json")))
    assert g["mismatches"] == 0 and g["cases_checked"] >= 251032 and len(g["kat"]) >= 1480
    seen = set()
    for case in g["kat"]:
        inp = np.array(case["in"], np.uint32).view(np.float32)
        want = np.array(case["out"], np.uint32)
        if case["fn"].startswith("filterTable"):          # ImageBlock's tabulation of the reference's filter bodies: the table builders are ours
            kind = case["fn"][len("filterTable"):].lower()
            kw = {"gaussian": dict(radius=float(inp[0]), stddev=float(inp[1])), "mitchell": dict(radius=float(inp[0]), B=float(inp[1]), Cc=float(inp[2])), "tent": {}, "box": {}}[kind]
            r, tab = scenes.pk.filter_table(kind, **kw)
            assert np.float32(r) == inp[0] and np.array_equal(np.asarray(tab, np.float32).view(np.uint32), want), case["fn"]
            seen.add(case["fn"])
            continue
        got = kzo.math_probe(case["fn"], inp).view(np.uint32)
        assert np.array_equal(got, want), (case["fn"], inp.tolist())
        seen.add(case["fn"])
    assert len(seen) == 46 and {"kissEval", "kissPdf", "kissSample", "sampleVNDF", "dpdfSample", "samplerStratified", "samplerCorrelated",
                                "extraEval", "extraPdf", "extraSample", "texColorRamp", "texBlend", "texBackgroundUV", "texBackgroundDir", "sceneBackground", "pmj02bnTileSize"} <= seen
