"""Primary-hit hints (kz_trav_seed, kz_traverse.h): a traversal that starts from a preset best hit -- on the device, the triangle the
ray's pixel hit last (KzExtendJob<true>::seed) -- must return the same closest hit, bit for bit, whatever the hint is.  The host
emulation runs the very traversal code; the GPU tests render with the hints off and on."""
import numpy as np
import pytest

import scenes
import pykazen as pk

INVALID = 0xFFFFFFFF


def _camera_rays(E, desc, per_axis=48, seed=5):
    """primary rays of the scene's own camera through a jittered grid of pixel sample positions"""
    w, h = desc.camera.width, desc.camera.height
    rng = np.random.default_rng(seed)
    xs, ys = np.meshgrid((np.arange(per_axis) + 0.5) * w / per_axis, (np.arange(per_axis) + 0.5) * h / per_axis)
    s4 = np.zeros((per_axis * per_axis, 4), np.float32)
    s4[:, 0] = xs.ravel() + rng.uniform(-0.5, 0.5, xs.size)
    s4[:, 1] = ys.ravel() + rng.uniform(-0.5, 0.5, ys.size)
    s4[:, 2:] = 0.5
    return E.camera_rays(s4)


def _seed_emu(desc):
    import seed_emu
    return seed_emu.SeedEmu(desc)


def _seeds(geom, prim):
    return np.stack([np.asarray(geom, np.uint32), np.asarray(prim, np.uint32)], axis=1)


def _same(E, rays, ref, seeds):
    got, k = E.trace_seeded(rays, seeds)
    assert got.tobytes() == ref.tobytes()
    return k


SCENES = {
    "soup": lambda: scenes.big_scene(20000, 96, 64, 16),
    "cornell": lambda: scenes.cornell_scene(64, 64, 4),
    "studio": lambda: scenes.studio_scene(128, 128, 4),
}


@pytest.mark.parametrize("name", sorted(SCENES))
def test_seeded_trace_is_bit_exact(emu, name):
    sb = SCENES[name]()
    d = sb.desc()
    E = _seed_emu(d)
    rays = _camera_rays(E, d)
    ref = E.trace(rays)
    hit = ref["geom_id"] != INVALID
    assert hit.mean() > 0.3
    n_tris = np.array([d.meshes[g].n_triangles for g in range(d.n_meshes)], np.int64)

    # the right triangle: every hint is taken, the hits do not change
    assert _same(E, rays, ref, _seeds(ref["geom_id"], ref["prim_id"])) == int(hit.sum())
    # the hit of the neighbouring sample (what a pixel's previous sample usually hit)
    _same(E, rays, ref, _seeds(np.roll(ref["geom_id"], 1), np.roll(ref["prim_id"], 1)))
    # the neighbouring triangle of the same mesh
    g = np.where(hit, ref["geom_id"], 0).astype(np.int64)
    p = np.where(hit, ref["prim_id"], 0).astype(np.int64)
    _same(E, rays, ref, _seeds(g, (p + 1) % n_tris[g]))
    # a triangle the ray does hit, but behind its closest hit: taken as the seed, then beaten by the closest one
    behind = rays.copy()
    behind["tmin"] = np.where(hit, np.nextafter(ref["t"], np.float32(np.inf)), behind["tmin"])
    second = E.trace(behind)
    k = _same(E, rays, ref, _seeds(second["geom_id"], second["prim_id"]))
    if name != "cornell":          # the closed box has a second surface behind most hits, the open scenes behind some
        assert k > 0
    # triangles the ray misses (hits of far-away samples, mostly missed)
    _same(E, rays, ref, _seeds(ref["geom_id"][::-1], ref["prim_id"][::-1]))
    # indices out of range: no seed at all
    nm = d.n_meshes
    for gg, pp in ((nm, 0), (INVALID, 0), (0, int(n_tris[0])), (0, INVALID), (INVALID, INVALID)):
        assert _same(E, rays, ref, _seeds(np.full(len(rays), gg), np.full(len(rays), pp))) == 0
    E.close()


def test_seed_with_the_right_triangle_saves_node_steps(emu):
    """the point of the hint: with the closest hit preset, the node step culls with its t from the root on"""
    sb = scenes.big_scene(20000, 96, 64, 16)
    d = sb.desc()
    E = _seed_emu(d)
    rays = _camera_rays(E, d)
    ref = E.trace(rays)
    none = _seeds(np.full(len(rays), INVALID), np.zeros(len(rays)))
    plain = E.trace_stats(rays, none)
    seeded = E.trace_stats(rays, _seeds(ref["geom_id"], ref["prim_id"]))
    assert seeded["nodes"] < 0.9 * plain["nodes"], (plain, seeded)
    E.close()


def test_seeded_ties_resolve_by_ids(emu):
    """a hint at exactly the closest t but with a larger (geomID, primID) loses the tie, as it would without the hint"""
    from test_gpu_parity import _tie_scene
    sb = _tie_scene()
    E = _seed_emu(sb.desc())
    rays = scenes.primary_rays(64, 40.0, (0, 0, -3.0))
    ref = E.trace(rays)
    hit = ref["geom_id"] != INVALID
    assert hit.any() and (ref["geom_id"][hit] == 0).all()
    n = len(rays)
    # geom 0 prim 1, geom 1 prim 0 and geom 2 prims 0 and 1 are the same triangle
    for gg, pp in ((0, 1), (1, 0), (2, 0), (2, 1)):
        assert _same(E, rays, ref, _seeds(np.full(n, gg), np.full(n, pp))) > 0
    E.close()


# ---------------------------------------------------------------------------------------------------------------- GPU
def _render_twice(sb, builder, rect=None):
    G = pk.Gpu(sb.desc(), devices=(0,), builder=builder)
    out = {}
    for on in (0, 1, 0, 1):         # the second pass of each setting starts from the hints the first left behind
        G.configure("primary_hint", 2 * on)         # 2: whatever the scene's size
        G.stats(reset=True)
        f = G.render(rect=rect)
        out.setdefault(on, []).append((f, G.stats(reset=True)))
    G.close()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name,builder", [("cornell", pk.BUILD_HOST_SAH), ("studio", pk.BUILD_HOST_SAH), ("soup", pk.BUILD_LBVH)])
def test_primary_hint_renders_the_same_frame(gpu_lib, name, builder):
    sb = {"cornell": lambda: scenes.cornell_scene(64, 64, 16, with_texture=True, normalmap=True),
          "studio": lambda: scenes.studio_scene(128, 128, 16),
          "soup": lambda: scenes.big_scene(200000, 192, 108, 16)}[name]()
    out = _render_twice(sb, builder)
    f_off, s_off = out[0][1]
    for f, s in (out[1][0], out[1][1]):
        # the same paths with the same hits: the same counts, and frames that differ only by the order of the atomic splats
        for key in ("paths", "rays_extension", "rays_shadow", "vertices"):
            assert s[key] == s_off[key], key
        np.testing.assert_allclose(f, f_off, rtol=1e-5, atol=1e-5 * float(np.abs(f_off).max()))
        assert abs(float(f[..., :3].sum()) / float(f_off[..., :3].sum()) - 1.0) < 1e-6
    assert s_off["rays_seeded"] == 0 and out[0][0][1]["rays_seeded"] == 0
    # a small frame is one launch whose primary rays all start before the first ones end: its first render finds few hints, the
    # second finds the ones the first left behind
    assert out[1][0][1]["rays_seeded"] <= out[1][0][1]["paths"]
    assert 0 < out[1][1][1]["rays_seeded"] <= out[1][1][1]["paths"]


@pytest.mark.gpu
def test_primary_hint_rectangles_and_options(gpu_lib):
    """rectangles that do not cover whole 8x4 tiles (k_raygen's padding lanes), and the option's range"""
    sb = scenes.cornell_scene(61, 37, 8)
    G = pk.Gpu(sb.desc(), devices=(0,), builder=pk.BUILD_LBVH)
    G.configure("primary_hint", 0)
    ref = G.render(rect=(3, 5, 58, 30))
    assert G.stats()["rays_seeded"] == 0
    G.configure("primary_hint", 1)          # by scene size: this one is far too small
    G.render(rect=(3, 5, 58, 30))
    assert G.stats()["rays_seeded"] == 0
    G.configure("primary_hint", 2)
    G.render(rect=(3, 5, 58, 30))
    f = G.render(rect=(3, 5, 58, 30))
    np.testing.assert_allclose(f, ref, rtol=1e-5, atol=1e-5 * float(np.abs(ref).max()))
    assert G.stats()["rays_seeded"] > 0
    with pytest.raises(RuntimeError):
        G.configure("primary_hint", 3)
    G.close()
