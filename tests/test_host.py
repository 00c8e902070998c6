"""The C++ host (nano-kazen_b200/host): kazen's XML scene format and plugin registry above the C ABI.
CPU tests check parsing/flattening against numpy restatements and feed the flattened tables to the
oracle; the GPU tests render the same XML through the `path_mis` / `gpu_bvh` plugins."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

import pykazen as pk
import scenes

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BOX = os.path.join(HERE, "data", "box", "box.xml")
KAZEN = os.path.join(ROOT, "nano-kazen_b200", "host", "kazen")
SHIPPED_SCENES = os.path.join(HERE, "data", "kazen_scenes", "2022_q1")      # byte copies of two reference scenes (inputs, see the README there)
WARM = os.path.join(SHIPPED_SCENES, "WarmStudio", "WarmStudio.xml")
PARAM = os.path.join(SHIPPED_SCENES, "parameters", "default_m0_r0.5.xml")


@pytest.fixture(scope="module")
def host():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "nano-kazen_b200", "host")])
    return pk


def _np(ptr, n, dtype):
    return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(dtype)), shape=(n,)).copy()


def test_registered_plugin_names(host):
    names = set(host.host_registered_plugins())
    # every plugin on the hot path keeps kazen's registered name (SURVEY Appendix D); gpu_bvh is the new accel plugin
    for n in ("scene obj diffuse kazenstandard normalmap area perspective thinlens independent stratified correlated pmj02bn "
              "constanttexture imagetexture background colorramp blend gaussian mitchell tent box path_mis gpu_bvh "
              "dielectric mirror lambertian ggx roughconductor roughplastic roughdielectric normals ao whitted path_mats").split():
        assert n in names


def test_box_scene_flattening(host):
    hs = host.HostScene(BOX)
    d = hs.desc
    assert d.n_meshes == 3 and d.n_lights == 1 and d.n_images == 3
    assert d.camera.type == pk.CAM_THINLENS and (d.camera.width, d.camera.height) == (48, 32)
    assert abs(d.camera.aperture_radius - 0.02) < 1e-7 and abs(d.camera.focus_distance - 3.4) < 1e-6
    # stratified rounds 10 up to 16 = 4x4 (sampler.cpp:83-93)
    assert (d.sampler.type, d.sampler.sample_count, d.sampler.res_x, d.sampler.seed) == (pk.SAMPLER_STRATIFIED, 16, 4, 1)
    assert (d.integrator.max_depth, d.integrator.regularization) == (4, 1) and abs(d.integrator.trace_bias - 1e-3) < 1e-9
    # mitchell default radius 2, tabulated like block.cpp:13-21
    r, tab = pk.filter_table("mitchell")
    assert d.filter.radius == r and np.allclose(np.array(list(d.filter.table), np.float32), tab, rtol=2e-6, atol=1e-7)
    # camera matrices: lookat (parser.cpp:273-287) and perspective (camera.cpp:35-62)
    assert np.allclose(np.array(list(d.camera.camera_to_world)).reshape(4, 4), pk.lookat((0, 0, -3.4), (0, 0, 0), (0, 1, 0)), atol=1e-6)
    assert np.allclose(np.array(list(d.camera.sample_to_camera)).reshape(4, 4), pk.perspective_sample_to_camera(48, 32, 39.0, 0.1, 100.0), rtol=1e-4, atol=1e-5)
    # room: 5 quads -> 10 triangles split (0,1,2),(3,0,2), 8 de-duplicated vertices, no normals/uvs
    room = d.meshes[0]
    assert (room.n_vertices, room.n_triangles) == (8, 10) and not room.normals and not room.uvs
    F = _np(room.indices, 30, C.c_uint32).reshape(-1, 3)
    assert F[:2].tolist() == [[0, 1, 2], [3, 0, 2]] and F[2:4].tolist() == [[4, 5, 6], [7, 4, 6]]
    # sphere: transform ops apply in document order: scale, then rotate, then translate
    sph = d.meshes[1]
    V = _np(sph.positions, 3 * sph.n_vertices, C.c_float).reshape(-1, 3)
    N = _np(sph.normals, 3 * sph.n_vertices, C.c_float).reshape(-1, 3)
    assert np.allclose(V.mean(0), (-0.3, -0.55, 0.2), atol=0.03)
    assert np.allclose(np.linalg.norm(V - np.array((-0.3, -0.55, 0.2)), axis=1), 0.45, atol=1e-5)
    assert np.allclose(np.linalg.norm(N, axis=1), 1.0, atol=1e-5)
    assert np.allclose((V - np.array((-0.3, -0.55, 0.2), np.float32)) / 0.45, N, atol=1e-5)       # normals follow the rotation
    # first sphere vertex is the +y pole (rotation about y leaves it in place)
    assert np.allclose(V[0], (-0.3, -0.1, 0.2), atol=1e-5)
    # materials: normalmap(kiss(blend, colorramp, constant)); light radiance = intensity * color
    outer = d.bsdfs[d.meshes[1].bsdf]
    assert outer.type == pk.BSDF_NORMALMAP and d.bsdfs[outer.nested].type == pk.BSDF_KISS
    kiss = d.bsdfs[outer.nested]
    assert d.textures[kiss.base_color].type == pk.TEX_BLEND and d.textures[kiss.roughness].type == pk.TEX_COLORRAMP
    assert abs(kiss.clearcoat - 0.5) < 1e-7 and abs(kiss.specular - 0.5) < 1e-7 and abs(kiss.sheen_tint - 0.5) < 1e-7
    assert d.textures[outer.normal_map].srgb == 0 and abs(d.textures[outer.normal_map].scale - 3.0) < 1e-7
    assert np.allclose(list(d.lights[0].radiance), (12.0, 10.8, 8.4), rtol=1e-6) and d.lights[0].primary_visibility == 0
    assert d.background >= 0 and d.textures[d.background].type == pk.TEX_BACKGROUND
    # PNG decode: row 0 = first scanline, values /255
    im = d.images[d.textures[d.textures[kiss.base_color].child[1]].image]
    assert (im.width, im.height) == (32, 16)
    px = _np(im.rgb, 3 * 32 * 16, C.c_float).reshape(16, 32, 3)
    rng = np.random.default_rng(3)
    assert np.allclose(px, rng.integers(30, 230, (16, 32, 3), dtype=np.uint8) / 255.0, atol=1e-6)
    assert hs.accel_builder() == pk.BUILD_HOST_SAH
    hs.close()


def test_overrides_and_defaults(host):
    hs = host.HostScene(BOX, {"camera.width": "i:20", "camera.height": "i:10", "sampler.type": "s:correlated", "sampler.sampleCount": "i:7",
                              "scene.accelBuilder": "s:lbvh", "integrator.maxDepth": "i:2"})
    d = hs.desc
    assert (d.camera.width, d.camera.height) == (20, 10)
    # correlated: res.y = (int)sqrt(7) = 2, res.x = ceil(7/2) = 4, spp = 8 (sampler.cpp:178-189)
    assert (d.sampler.type, d.sampler.sample_count, d.sampler.res_x, d.sampler.res_y) == (pk.SAMPLER_CORRELATED, 8, 4, 2)
    assert d.integrator.max_depth == 2 and hs.accel_builder() == pk.BUILD_LBVH
    hs.close()


@pytest.mark.parametrize("xml,msg", [
    ("<scene><foo/></scene>", "unexpected tag"),
    ("<scene><integer name='a'/></scene>", "missing attribute"),
    ("<scene><integer name='a' value='1' extra='2'/></scene>", "unexpected attribute"),
    ("<scene><integrator type='nope'/></scene>", "could not be found"),
    ("<scene><camera type='gaussian'/></scene>", "Unexpectedly constructed"),
    ("<scene><translate value='1 2 3'/></scene>", "transform nodes"),
    ("<scene><integrator type='path_mis'/></scene>", "No camera was specified"),
    ("<scene><camera type='perspective'/></scene>", "No integrator was specified"),
    ("<scene><float name='x' value='abc'/></scene>", "Could not parse floating point"),
    ("<float name='x' value='1'/>", "must be a kazen object"),
    ("<scene><integrator type='path_mis'/><camera type='perspective'/><mesh type='obj'><string name='filename' value='missing.obj'/></mesh></scene>", "Unable to open OBJ"),
    ("<scene><mesh type='obj'></scene>", "mismatched closing tag"),
])
def test_parser_errors(host, tmp_path, xml, msg):
    p = tmp_path / "bad.xml"
    p.write_text(xml)
    with pytest.raises(RuntimeError, match=msg):
        host.HostScene(str(p))


def test_host_tables_feed_the_oracle(host, kzo):
    """XML -> plugins -> POD tables -> oracle render: the same tables the GPU would receive are a valid,
    lit scene; the numpy-built twin of the scene (pykazen.SceneBuilder) renders the same image."""
    hs = host.HostScene(BOX)
    O = kzo.Oracle(hs.desc)
    f = O.render()
    rgb, _ = O.resolve(f)
    assert np.isfinite(rgb).all() and 0.05 < rgb.mean() < 2.0
    st = O.stats()
    assert st["paths"] == 48 * 32 * 16 and st["rays_shadow"] > 0
    O.close(); hs.close()


def test_fallback_pmj_tables_are_stratified(host):
    """the stand-in tables keep the one property the PMJ02BN constructor relies on (sampler.cpp:290-314):
    the first 65536 points of set 0 put exactly spp points into every pixel-tile cell"""
    bn, pm = host.host_fallback_tables()
    assert bn.shape == (48, 128, 128) and pm.shape == (5, 65536, 2)
    p = pm[0].astype(np.float64) * 2.0 ** -32
    for spp in (1, 4, 16, 64):
        T = 1 << (8 - int(round(np.log(spp) / np.log(4))))
        cells = (np.floor(p[:, 0] * T) + T * np.floor(p[:, 1] * T)).astype(np.int64)
        assert (np.bincount(cells, minlength=T * T) == spp).all()
    # every set is a (0,2)-net in base 2 over its first 4096 points: 64x64, 4096x1 and 1x4096 grids all hit once
    for s in range(5):
        q = pm[s, :4096].astype(np.float64) * 2.0 ** -32
        for (a, b) in ((64, 64), (4096, 1), (1, 4096), (16, 256)):
            idx = (np.floor(q[:, 0] * a) * b + np.floor(q[:, 1] * b)).astype(np.int64)
            assert len(np.unique(idx)) == 4096


def test_extra_bsdf_plugins_from_xml(host, tmp_path):
    """SURVEY 8(f)-1 plugins keep kazen's property names and defaults (bsdf.cpp:100-106,632-633,696-714,818-842,951-961)"""
    (tmp_path / "q.obj").write_text("v -1 -1 0\nv 1 -1 0\nv 1 1 0\nv -1 1 0\nf 1 2 3 4\n")
    bs = ['<bsdf type="dielectric"/>', '<bsdf type="dielectric"><float name="intIOR" value="1.33"/></bsdf>', '<bsdf type="mirror"/>',
          '<bsdf type="lambertian"><texture type="constanttexture"><color name="color" value="0.1 0.2 0.3"/></texture></bsdf>',
          '<bsdf type="ggx"><float name="roughness" value="0.3"/><texture type="constanttexture"/></bsdf>',
          '<bsdf type="roughconductor"><string name="material" value="Cu"/><float name="alpha" value="0.2"/></bsdf>',
          '<bsdf type="roughplastic"><color name="kd" value="0.2 0.3 0.4"/></bsdf>', '<bsdf type="roughdielectric"/>']
    xml = "<scene><integrator type='path_mis'/><camera type='perspective'/>" + "".join(
        f"<mesh type='obj'><string name='filename' value='q.obj'/>{b}</mesh>" for b in bs) + "</scene>"
    (tmp_path / "s.xml").write_text(xml)
    hs = host.HostScene(str(tmp_path / "s.xml"))
    d = hs.desc
    B = [d.bsdfs[d.meshes[i].bsdf] for i in range(d.n_meshes)]
    assert [b.type for b in B] == [pk.BSDF_DIELECTRIC, pk.BSDF_DIELECTRIC, pk.BSDF_MIRROR, pk.BSDF_LAMBERTIAN, pk.BSDF_GGX, pk.BSDF_ROUGHCONDUCTOR,
                                   pk.BSDF_ROUGHPLASTIC, pk.BSDF_ROUGHDIELECTRIC]
    assert abs(B[0].int_ior - 1.5046) < 1e-6 and abs(B[0].ext_ior - 1.000277) < 1e-6 and abs(B[1].int_ior - 1.33) < 1e-6
    assert d.textures[B[3].base_color].type == pk.TEX_CONSTANT and abs(d.textures[B[3].base_color].color[1] - 0.2) < 1e-7
    assert abs(B[4].alpha - 0.3) < 1e-7 and B[4].anisotropy == 0.0
    assert abs(B[5].alpha - 0.04) < 1e-7 and np.allclose(list(B[5].eta), pk.CONDUCTORS["Cu"][0]) and np.allclose(list(B[5].k), pk.CONDUCTORS["Cu"][1])
    assert abs(B[6].alpha - 0.01) < 1e-7 and np.allclose(list(B[6].albedo), (0.2, 0.3, 0.4))
    assert abs(B[7].alpha - 0.01) < 1e-7
    hs.close()
    (tmp_path / "bad.xml").write_text(xml.replace('value="Cu"', 'value="Zz"'))
    with pytest.raises(RuntimeError, match="unknown material"):
        host.HostScene(str(tmp_path / "bad.xml"))


def test_cli_fails_loudly_without_gpu(host, tmp_path):
    """run where no device is visible, so that the check holds on GPU machines as well"""
    r = subprocess.run([KAZEN, BOX, "-o", str(tmp_path / "box")], capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode != 0 and "no CUDA device" in r.stderr and "no CPU fallback" in r.stderr


def test_reference_scenes_parse_unchanged(host, kzo):
    """kazen's own scene files as tests/data/kazen_scenes ships them (WarmStudio + the default parameter-sweep scene) load unchanged
    through the plugin system"""
    xmls = [WARM, PARAM]
    tris = {}
    for x in xmls:
        hs = host.HostScene(x, {"camera.width": "i:64", "camera.height": "i:36"})
        d = hs.desc
        tris[os.path.basename(x)] = sum(d.meshes[i].n_triangles for i in range(d.n_meshes))
        assert d.sampler.type == pk.SAMPLER_INDEPENDENT and d.n_lights >= 1
        hs.close()
    assert tris["WarmStudio.xml"] == 17952 and tris["default_m0_r0.5.xml"] == 36378      # SURVEY 0 / 8d
    # WarmStudio through the oracle at low resolution: the loose golden anchor of BASELINE.md (shipped PNG mean)
    hs = host.HostScene(xmls[0], {"camera.width": "i:96", "camera.height": "i:54", "sampler.type": "s:stratified", "sampler.sampleCount": "i:16"})
    O = kzo.Oracle(hs.desc)
    _, srgb = O.resolve(O.render())
    m = srgb.reshape(-1, 3).mean(0)
    assert 20 < m[0] < 45 and 14 < m[1] < 34 and 5 < m[2] < 18 and m[0] > m[1] > m[2]       # shipped PNG: (36.5, 27.5, 13.1)
    O.close(); hs.close()
    # the default parameter-sweep scene against the mean of the reference's golden PNG of it (8-bit and older than the Q2
    # changes, so the frame mean sits up to ~0.045 lower here)
    hs = host.HostScene(xmls[1], {"camera.width": "i:192", "camera.height": "i:108", "sampler.sampleCount": "i:36", "sampler.type": "s:stratified"})
    O = kzo.Oracle(hs.desc)
    rgb, _ = O.resolve(O.render())
    d = np.minimum(rgb, 1.0).mean(axis=(0, 1)) - np.array(_golden_means()["default_m0_r0.5"])
    assert (-0.045 < d).all() and (d < 0.005).all(), d
    O.close(); hs.close()


def test_shipped_scene_fixtures_are_the_reference_files():
    """tests/data/kazen_scenes holds byte copies of the reference's scene files (so that 'an existing scene file renders unchanged');
    tests/golden/kazen_scenes_sha256.json holds the SHA-256 of each reference file, taken when the copies were compared byte for byte
    with the reference tree"""
    import hashlib
    gold = json.load(open(os.path.join(HERE, "golden", "kazen_scenes_sha256.json")))
    got = {}
    for root, _, files in os.walk(SHIPPED_SCENES):
        for f in files:
            p = os.path.join(root, f)
            got[os.path.relpath(p, SHIPPED_SCENES)] = hashlib.sha256(open(p, "rb").read()).hexdigest()
    assert got == gold
    assert len(got) == 11


def test_shipped_scenes_parse(host, kzo):
    """the two fixtures SURVEY 8(d)-1 names, through the plugin system: triangle counts, emitters, filters"""
    hs = host.HostScene(WARM)
    d = hs.desc
    assert sum(d.meshes[i].n_triangles for i in range(d.n_meshes)) == 17952 and d.n_lights == 1 and d.meshes[2].n_triangles == 32
    assert (d.camera.width, d.camera.height) == (1920, 1080) and d.sampler.sample_count == 40 and abs(d.filter.radius - 2.0) < 1e-7
    hs.close()
    hs = host.HostScene(PARAM)
    d = hs.desc
    assert sum(d.meshes[i].n_triangles for i in range(d.n_meshes)) == 36378 and d.n_lights == 3
    hs.close()


@pytest.fixture(scope="module")
def config_scenes(tmp_path_factory):
    """BASELINE configs[2] / configs[3] stand-ins at test size (512^2 textures, 96 x 48 ball), see tests/data/make_configs.py"""
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_configs", os.path.join(HERE, "data", "make_configs.py"))
    mc = importlib.util.module_from_spec(spec); spec.loader.exec_module(mc)
    return mc.generate(str(tmp_path_factory.mktemp("kzcfg")), tex_res=512, ball=(96, 48))


def test_config_scenes_parse(host, config_scenes):
    hs = host.HostScene(os.path.join(config_scenes, "c3_lookdev_4k.xml"))
    d = hs.desc
    assert d.camera.type == pk.CAM_THINLENS and (d.camera.width, d.camera.height) == (3840, 2160) and d.n_lights == 3
    types = sorted(d.bsdfs[i].type for i in range(d.n_bsdfs))
    assert pk.BSDF_NORMALMAP in types and pk.BSDF_KISS in types
    assert d.n_images == 3 and d.images[0].width == 512
    ttypes = [d.textures[i].type for i in range(d.n_textures)]
    assert pk.TEX_BLEND in ttypes and ttypes.count(pk.TEX_IMAGE) == 3
    hs.close()
    hs = host.HostScene(os.path.join(config_scenes, "c4_pmj02bn_1080p.xml"))
    d = hs.desc
    assert d.sampler.type == pk.SAMPLER_PMJ02BN and d.integrator.regularization == 1 and abs(d.integrator.accumulated_roughness - 0.5) < 1e-7
    assert (d.camera.width, d.camera.height) == (1920, 1080) and d.n_meshes == 6
    assert d.meshes[5].n_triangles == 12 * 6 * 2 - 2 * 12 and bool(d.meshes[5].normals)      # the low-poly smooth sphere
    hs.close()


# --------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("which,size,spp", [("c3_lookdev_4k", (240, 135), 16), ("c4_pmj02bn_1080p", (240, 135), 16)])
def test_gpu_renders_config_scenes_like_oracle(host, kzo, gpu_lib, config_scenes, which, size, spp):
    """configs[2] (thin lens + normal map + image textures through blend) and configs[3] (pmj02bn + regularisation + traceBias +
    low-poly smooth sphere) through the XML host: GPU vs oracle at equal samples, both accel builders."""
    ov = {"camera.width": f"i:{size[0]}", "camera.height": f"i:{size[1]}", "sampler.sampleCount": f"i:{spp}"}
    hs = host.HostScene(os.path.join(config_scenes, which + ".xml"), ov)
    O = kzo.Oracle(hs.desc)
    ro, _ = O.resolve(O.render())
    assert ro.mean() > 0.05
    for builder in (pk.BUILD_HOST_SAH, pk.BUILD_LBVH):
        G = pk.Gpu(hs.desc, builder=builder)
        rg, _ = G.resolve(G.render())
        st = G.stats()
        assert scenes.rel_mse(rg, ro).max() < 2e-4
        assert st["paths"] == size[0] * size[1] * spp and st["rays_shadow"] > 0
        G.close()
    O.close(); hs.close()


def _golden_means():
    import json
    return json.load(open(os.path.join(HERE, "golden", "param_means.json")))


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["WarmStudio", "default_m0_r0.5"])
def test_gpu_renders_kazens_own_scene_files(host, kzo, gpu_lib, which, tmp_path):
    """north_star: 'an existing scene file renders unchanged with the GPU integrator and accelerator selected as plugins'.
    (1) configs[0]: the file at 512x512, 64 spp, stratified -- GPU image vs the oracle at equal samples (relMSE);
    (2) the `kazen` CLI on the very file (its own resolution scaled down, its own independent sampler): mean linear RGB against
        the reference's shipped 1920x1080 PNG of that file (BASELINE.md section 2 gate: |delta| <= 0.02 per channel; the goldens
        predate the Q2 changes, which is what the 0.045 on the bright parameter scene allows for)."""
    xml = WARM if which == "WarmStudio" else PARAM
    ov = {"camera.width": "i:512", "camera.height": "i:512", "sampler.type": "s:stratified", "sampler.sampleCount": "i:64"}
    hs = host.HostScene(xml, ov)
    G = pk.Gpu(hs.desc, builder=hs.accel_builder())
    O = kzo.Oracle(hs.desc)
    fg = G.render()
    rg, _ = G.resolve(fg)
    st = G.stats()
    assert st["paths"] == 512 * 512 * 64
    # the oracle renders 16 of the 64 sample indices of the same frame (the CPU port needs ~6 s for all of them on 16 cores;
    # equal-sample parity is on that range, the full GPU frame must agree with it as a noisier estimate of the same image)
    fo = O.render(0, 16)
    ro, _ = O.resolve(fo)
    rg16, _ = G.resolve(G.render(0, 16))
    assert scenes.rel_mse(rg16, ro).max() < 2e-4
    assert abs(rg.mean() - ro.mean()) < 0.02 * max(ro.mean(), 0.02)
    O.close(); G.close(); hs.close()
    out = str(tmp_path / which)
    r = subprocess.run([KAZEN, xml, "-o", out, "--size", "480x270", "--spp", "64"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    from PIL import Image
    png = np.asarray(Image.open(out + ".png")).astype(np.float64) / 255.0
    lin = np.where(png <= 0.04045, png / 12.92, ((png + 0.055) / 1.055) ** 2.4).mean(axis=(0, 1))
    gold = np.array(_golden_means()[which])
    tol = 0.02 if which == "WarmStudio" else 0.045
    assert np.abs(lin - gold).max() < tol, (lin, gold)


@pytest.mark.gpu
def test_gpu_renders_xml_scene_like_oracle(host, kzo, gpu_lib):
    hs = host.HostScene(BOX)
    O = kzo.Oracle(hs.desc)
    G = pk.Gpu(hs.desc, builder=hs.accel_builder())
    ro, _ = O.resolve(O.render()); rg, _ = G.resolve(G.render())
    assert scenes.rel_mse(rg, ro).max() < 2e-4
    O.close(); G.close(); hs.close()


@pytest.mark.gpu
def test_kazen_cli_on_gpu(host, kzo, tmp_path):
    """kazen <scene.xml>: the XML renders through the path_mis / gpu_bvh plugins and writes a PNG + raw frame"""
    out = str(tmp_path / "box")
    r = subprocess.run([KAZEN, BOX, "-o", out, "--raw", "--accel", "lbvh"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "Render ready" in r.stdout and os.path.getsize(out + ".png") > 500
    raw = np.fromfile(out + ".rgbw", np.uint8)
    w, h, b = np.frombuffer(raw[:12].tobytes(), np.int32)
    frame = np.frombuffer(raw[12:].tobytes(), np.float32).reshape(h + 2 * b, w + 2 * b, 4)
    hs = host.HostScene(BOX)
    O = kzo.Oracle(hs.desc)
    ro, _ = O.resolve(O.render()); rg, _ = O.resolve(np.ascontiguousarray(frame))
    assert scenes.rel_mse(rg, ro).max() < 2e-4
    from PIL import Image
    png = np.asarray(Image.open(out + ".png"))
    _, so = O.resolve(np.ascontiguousarray(frame))
    assert png.shape == (h, w, 3) and np.abs(png.astype(int) - so.astype(int)).max() <= 1
    O.close(); hs.close()


def test_image_readers_reject_malformed_headers(host, tmp_path):
    """header fields of texture files are untrusted: out-of-range sizes, a missing IHDR and a channel list that runs past its
    attribute are errors, not out-of-bounds reads or huge allocations"""
    import struct, zlib

    def png(chunks):
        out = b"\x89PNG\r\n\x1a\n"
        for t, d in chunks:
            out += struct.pack(">I", len(d)) + t + d + struct.pack(">I", zlib.crc32(t + d) & 0xFFFFFFFF)
        return out
    idat = zlib.compress(b"\x00" + bytes(3))
    cases = {
        "huge.png": png([(b"IHDR", struct.pack(">IIBBBBB", 0xFFFFFFF0, 7, 8, 2, 0, 0, 0)), (b"IDAT", idat), (b"IEND", b"")]),
        "zero.png": png([(b"IHDR", struct.pack(">IIBBBBB", 0, 1, 8, 2, 0, 0, 0)), (b"IDAT", idat), (b"IEND", b"")]),
        "noihdr.png": png([(b"IDAT", idat), (b"IEND", b""), (b"tEXt", b"padding-padding-padding")]),
        "neg.pfm": b"PF\n-4 4\n-1.0\n" + bytes(64),
        "big.hdr": b"#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n\n-Y 2000000 +X 2000000\n",
    }
    # EXR: a channel list whose last name has no terminator inside the attribute
    exr = bytes([0x76, 0x2f, 0x31, 0x01, 2, 0, 0, 0]) + b"channels\0chlist\0" + struct.pack("<i", 3) + b"RGB" + b"compression\0compression\0" + struct.pack("<i", 1) + b"\0" + b"\0"
    cases["chlist.exr"] = exr + bytes(64)
    for name, blob in cases.items():
        p = tmp_path / name
        p.write_bytes(blob)
        with pytest.raises(RuntimeError):
            host.host_read_image(str(p))


def test_jpeg_decoder_matches_libjpeg(host, tmp_path):
    """imagetexture's JPEG path (the reference's look-dev material uses .jpg textures through OpenImageIO = libjpeg): baseline
    Huffman decode with libjpeg's default arithmetic (slow-integer IDCT, fancy upsampling, fixed-point YCbCr) -- bit identical to
    Pillow's libjpeg-turbo decode for 4:4:4 / 4:2:2 / 4:2:0 / grayscale, odd sizes, restart intervals, optimised tables."""
    from PIL import Image
    rng = np.random.default_rng(11)
    yy, xx = np.mgrid[0:83, 0:131]
    base = np.stack([127 + 120 * np.sin(xx / 9.0) * np.cos(yy / 7.0), 255 * (xx % 32 < 16) * (yy % 24 < 12), 2 * yy + 0.5 * xx], -1)
    img = np.clip(base + rng.normal(0, 12, base.shape), 0, 255).astype(np.uint8)           # smooth + hard edges + noise
    cases = [dict(quality=90, subsampling=0), dict(quality=75, subsampling=1), dict(quality=60, subsampling=2), dict(quality=95, subsampling=2, optimize=True),
             dict(quality=30, subsampling=2), dict(quality=85, subsampling=2, restart_marker_blocks=3), dict(quality=85, subsampling=1, restart_marker_rows=1)]
    n = 0
    for k, kw in enumerate(cases):
        for size in ((131, 83), (16, 16), (3, 5), (1, 1), (2, 9), (64, 48)):
            p = str(tmp_path / f"t{k}_{size[0]}x{size[1]}.jpg")
            try:
                Image.fromarray(img[:size[1], :size[0]]).save(p, **kw)
            except (TypeError, ValueError):
                continue                                                                 # an older Pillow without restart markers
            want = np.asarray(Image.open(p).convert("RGB"))
            got = host.host_read_image(p)
            assert got.shape == want.shape
            assert np.array_equal(np.rint(got * 255).astype(np.uint8), want), (kw, size)
            n += 1
    assert n >= 30
    p = str(tmp_path / "g.jpg")
    Image.fromarray(img[..., 0]).save(p, quality=80)
    want = np.asarray(Image.open(p))
    got = host.host_read_image(p)
    assert np.array_equal(np.rint(got[..., 0] * 255).astype(np.uint8), want) and np.array_equal(got[..., 0], got[..., 2])
    p = str(tmp_path / "prog.jpg")
    Image.fromarray(img).save(p, progressive=True)
    with pytest.raises(RuntimeError, match="progressive"):
        host.host_read_image(p)
    (tmp_path / "bad.jpg").write_bytes(open(str(tmp_path / "t0_131x83.jpg"), "rb").read()[:900])
    with pytest.raises(RuntimeError):
        host.host_read_image(str(tmp_path / "bad.jpg"))


@pytest.mark.gpu
def test_kazen_cli_resumes_a_render(host, tmp_path):
    """Progressive / resumable accumulation (SURVEY 8f-4): sample indices [0, A) saved as a raw frame, [A, N) added to it by a second
    process; the sum is the one-shot render up to the order of the float additions."""
    def load(stem):
        raw = np.fromfile(stem + ".rgbw", np.uint8)
        w, h, b = np.frombuffer(raw[:12].tobytes(), np.int32)
        return np.frombuffer(raw[12:].tobytes(), np.float32).reshape(h + 2 * b, w + 2 * b, 4)
    full, part, rest = (str(tmp_path / n) for n in ("full", "part", "rest"))
    for args in (["-o", full, "--raw"], ["-o", part, "--raw", "--spp-range", "0:5"], ["-o", rest, "--raw", "--spp-range", "5:9999", "--resume", part + ".rgbw"]):
        r = subprocess.run([KAZEN, BOX] + args, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    a, c = load(full), load(rest)
    assert not np.array_equal(load(part), a)
    assert np.allclose(a, c, rtol=1e-4, atol=1e-5)
    r = subprocess.run([KAZEN, BOX, "-o", rest, "--size", "33x17", "--resume", part + ".rgbw"], capture_output=True, text=True)
    assert r.returncode != 0 and "does not match" in r.stderr


def test_image_readers(host, tmp_path):
    """imagetexture decoders of the host: PNG, PFM, Radiance HDR, scanline OpenEXR (NONE / RLE / ZIPS / ZIP, HALF / FLOAT)"""
    os.environ["OPENCV_IO_ENABLE_OPENEXR"] = "1"
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(8)
    img = rng.uniform(0.0, 4.0, (19, 37, 3)).astype(np.float32)          # odd sizes: ZIP blocks of 16 lines with a ragged tail
    bgr = np.ascontiguousarray(img[..., ::-1])
    for comp in (cv2.IMWRITE_EXR_COMPRESSION_NO, cv2.IMWRITE_EXR_COMPRESSION_RLE, cv2.IMWRITE_EXR_COMPRESSION_ZIPS, cv2.IMWRITE_EXR_COMPRESSION_ZIP):
        for typ, tol in ((cv2.IMWRITE_EXR_TYPE_FLOAT, 0.0), (cv2.IMWRITE_EXR_TYPE_HALF, 2e-3)):
            p = str(tmp_path / f"t_{comp}_{typ}.exr")
            assert cv2.imwrite(p, bgr, [cv2.IMWRITE_EXR_COMPRESSION, comp, cv2.IMWRITE_EXR_TYPE, typ])
            got = host.host_read_image(p)
            assert got.shape == img.shape and np.allclose(got, img, rtol=tol, atol=tol * 4), (comp, typ)
    smooth = np.tile(np.linspace(0.1, 3.0, 64, dtype=np.float32)[None, :, None], (9, 1, 3))       # runs: exercises the HDR RLE path
    p = str(tmp_path / "t.hdr")
    assert cv2.imwrite(p, np.ascontiguousarray(smooth[..., ::-1]))
    got = host.host_read_image(p)
    assert got.shape == smooth.shape and np.allclose(got, smooth, rtol=1e-2)
    # PFM written by hand (bottom-to-top scanlines, little endian)
    p = str(tmp_path / "t.pfm")
    with open(p, "wb") as f:
        f.write(b"PF\n37 19\n-1.0\n"); f.write(img[::-1].tobytes())
    assert np.array_equal(host.host_read_image(p), img)
    with pytest.raises(RuntimeError, match="unsupported image format"):
        (tmp_path / "x.tif").write_bytes(b"II*\x00junk"); host.host_read_image(str(tmp_path / "x.tif"))
    # the host's own EXR writer (bitmap.cpp:23-36): read back by our reader and by an independent one (OpenCV)
    p = str(tmp_path / "w.exr")
    host.host_write_exr(p, img)
    assert np.array_equal(host.host_read_image(p), img)
    back = cv2.imread(p, cv2.IMREAD_UNCHANGED)
    assert back is not None and np.array_equal(back[..., ::-1], img)


def test_obj_loader_matches_the_reference_class(tmp_path):
    """tests/golden/obj_kat.json holds what the reference's OWN WavefrontOBJ class (mesh.cpp:200-343, compiled in place by
    oracle/ref_obj_kat.cpp) builds from tests/golden/obj/*.obj: vertex / normal / texture-coordinate / index arrays.  The C++ host's
    loader must produce the same arrays bit for bit: parsing (exponents, tabs, blank and foreign lines), quads split (0 1 2, 3 0 2),
    vertices de-duplicated by (position, texcoord, normal) index triple in order of first use, normals normalised, v//n and v/t forms."""
    import ctypes as C
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "obj_kat.json")))["files"]
    assert len(gold) >= 5
    for name, g in sorted(gold.items()):
        xml = tmp_path / (name + ".xml")
        xml.write_text(f"""<?xml version="1.0" ?>
<scene>
    <integrator type="path_mis"/>
    <sampler type="independent"><integer name="sampleCount" value="1"/></sampler>
    <camera type="perspective"><integer name="width" value="8"/><integer name="height" value="8"/></camera>
    <mesh type="obj"><string name="filename" value="{os.path.join(ROOT, 'tests', 'golden', 'obj', name)}"/><bsdf type="diffuse"/></mesh>
</scene>""")
        hs = pk.HostScene(str(xml))
        assert hs.desc.n_meshes == 1
        m = hs.desc.meshes[0]
        nv, nt = m.n_vertices, m.n_triangles
        V = np.ctypeslib.as_array(m.positions, (nv * 3,)).view(np.uint32)
        F = np.ctypeslib.as_array(m.indices, (nt * 3,))
        assert V.tolist() == g["V"], name
        assert F.tolist() == g["F"], name
        if g["N"]:
            assert np.ctypeslib.as_array(m.normals, (nv * 3,)).view(np.uint32).tolist() == g["N"], name
        else:
            assert not m.normals
        if g["UV"]:
            assert np.ctypeslib.as_array(m.uvs, (nv * 2,)).view(np.uint32).tolist() == g["UV"], name
        else:
            assert not m.uvs
        hs.close()
