"""Animation in place: kzgpu_mesh_update + kzgpu_accel_refit (kz_refit.h) and kzgpu_camera_update.

A refitted accel keeps the tree the build made for the old positions and gets new boxes and triangle records.  The traversal's hits do
not depend on the tree (culling is conservative, ties go to the smallest (t, geomID, primID)), so after a refit trace and occluded must
return exactly what the oracle returns on the moved scene.  The node bytes are held to a numpy restatement of the rule: k_collapse's
quantisation of the exact box of each slot's subtree -- tight and containing, so a conservative but useless refit fails too.
The CPU tests run the very refit code on the host emulation's accel (tests/hostemu/refit_emu.cpp); the GPU tests run the C ABI."""
import ctypes as C

import numpy as np
import pytest

import scenes
import pykazen as pk

INVALID = 0xFFFFFFFF
NODE_DTYPE = np.dtype([("p", "<f4", 3), ("e", "u1", 3), ("imask", "u1"), ("child_base", "<u4"), ("tri_base", "<u4"), ("trimask", "<u4"),
                       ("magic", "<u4"), ("qlo", "u1", (3, 8)), ("qhi", "u1", (3, 8))])
TOPOLOGY = ("imask", "child_base", "tri_base", "trimask", "magic")


# ------------------------------------------------------------------------------------------------------------ scenes and motion
def _positions(d, g):
    m = d.meshes[g]
    return np.ctypeslib.as_array(m.positions, shape=(m.n_vertices * 3,)).reshape(-1, 3).copy()


def _indices(d, g):
    m = d.meshes[g]
    return np.ctypeslib.as_array(m.indices, shape=(m.n_triangles * 3,)).reshape(-1, 3).copy()


def moved(d, positions, keep):
    """a copy of scene desc `d` whose meshes g in `positions` have the given vertex positions (`keep` holds the new arrays)"""
    dd = pk.SceneDesc.from_buffer_copy(d)
    meshes = (pk.MeshDesc * max(1, d.n_meshes))()
    for g in range(d.n_meshes):
        C.memmove(C.byref(meshes[g]), C.byref(d.meshes[g]), C.sizeof(pk.MeshDesc))
        if g in positions:
            P = np.ascontiguousarray(positions[g], np.float32).reshape(-1, 3)
            assert P.shape[0] == d.meshes[g].n_vertices
            keep.append(P)
            meshes[g].positions = P.ctypes.data_as(pk.c_float_p)
    dd.meshes = meshes
    keep += [meshes, dd]
    return dd


def _mean_edge(P, F):
    a, b, c = P[F[:, 0]], P[F[:, 1]], P[F[:, 2]]
    return float(np.mean([np.linalg.norm(b - a, axis=1).mean(), np.linalg.norm(c - b, axis=1).mean(), np.linalg.norm(a - c, axis=1).mean()]))


def _biggest(d, lights=False):
    ok = [g for g in range(d.n_meshes) if (d.meshes[g].light >= 0) == lights]
    return max(ok, key=lambda g: d.meshes[g].n_triangles)


def deform(d, kind, seed=1):
    """new positions {mesh: (n_vertices, 3) float32} for one of the motions the refit has to follow"""
    rng = np.random.default_rng(seed)
    all_p = np.concatenate([_positions(d, g) for g in range(d.n_meshes)])
    size = float(np.abs(all_p).max())
    g0 = _biggest(d)
    P, F = _positions(d, g0), _indices(d, g0)
    if kind == "jitter":             # every vertex of every mesh, about half a mean edge length of its mesh
        return {g: _positions(d, g) + rng.normal(0, 0.5 * _mean_edge(_positions(d, g), _indices(d, g)), (d.meshes[g].n_vertices, 3)).astype(np.float32)
                for g in range(d.n_meshes)}
    if kind == "translate":          # one mesh far away
        return {g0: P + np.array([7.0, -4.0, 5.0], np.float32) * np.float32(size)}
    if kind == "scale":              # one mesh 10^3 times larger: scene_max_abs grows with it
        c = P.mean(0)
        return {g0: (c + (P - c) * np.float32(1000.0)).astype(np.float32)}
    if kind == "collapse":           # a third of one mesh's triangles collapse to points, another third to segments
        k = F.shape[0] // 3
        Q = P.copy()
        Q[F[:k, 1]] = Q[F[:k, 0]]; Q[F[:k, 2]] = Q[F[:k, 0]]
        Q[F[k:2 * k, 2]] = Q[F[k:2 * k, 1]]
        return {g0: Q}
    if kind == "permute":            # vertices permuted: triangles cross the scene
        return {g: _positions(d, g)[rng.permutation(d.meshes[g].n_vertices)] for g in range(d.n_meshes) if d.meshes[g].light < 0}
    raise ValueError(kind)


MOTIONS = ("jitter", "translate", "scale", "collapse", "permute")
SCENES = {
    "soup": lambda: scenes.soup_scene(1 << 15),
    "cornell": lambda: scenes.cornell_scene(32, 32, 4),
    "studio": lambda: scenes.studio_scene(48, 48, 4),
}


def probe_rays(d, n=40000, seed=3):
    """incoherent rays over the scene's extent (a quarter of them short) and rays aimed at random points of random triangles, wherever
    the motion took them"""
    rng = np.random.default_rng(seed)
    tris = np.concatenate([_positions(d, g)[_indices(d, g)] for g in range(d.n_meshes) if d.meshes[g].n_triangles])
    lo, hi = tris.reshape(-1, 3).min(0), tris.reshape(-1, 3).max(0)
    r = np.zeros(2 * n, pk.RAY_DTYPE)
    o = rng.uniform(lo - 0.1 * (hi - lo), hi + 0.1 * (hi - lo), (2 * n, 3))
    dirs = rng.normal(size=(n, 3))
    target = tris[rng.integers(0, len(tris), n)]
    w = rng.dirichlet((1, 1, 1), n)
    aim = (target * w[:, :, None]).sum(1) - o[n:]
    dirs = np.concatenate([dirs, aim])
    dirs /= np.maximum(np.linalg.norm(dirs, axis=1, keepdims=True), 1e-30)
    r["o"] = o.astype(np.float32); r["d"] = dirs.astype(np.float32)
    r["tmin"] = np.float32(1e-4); r["tmax"] = np.inf
    r["tmax"][: n // 2] = (np.linalg.norm(hi - lo) * rng.uniform(0.05, 0.5, n // 2)).astype(np.float32)
    return r


# ------------------------------------------------------------------------------------------------------------ the rule, in numpy
def _popc(x):
    return np.bitwise_count(np.asarray(x, np.uint32)).astype(np.int64)


def refit_records(pre_tris, d):
    """the triangle records re-gathered from the positions of `d`: (n, 3, 4) float32, (geomID, primID) kept"""
    out = np.array(pre_tris, np.float32, copy=True).reshape(-1, 3, 4)
    geom = out[:, 0, 3].view(np.uint32).astype(np.int64); prim = out[:, 1, 3].view(np.uint32).astype(np.int64)
    for g in np.unique(geom):
        sel = geom == g
        pts = _positions(d, int(g))[_indices(d, int(g))[prim[sel]]]          # (k, 3, 3)
        out[sel, :, :3] = pts
    out[:, 2, 3] = 0.0
    return out


def node_levels(nodes):
    """node index arrays per level, root first (children of level l's internal slots form level l + 1)"""
    levels, cur = [], np.array([0], np.int64) if len(nodes) else np.zeros(0, np.int64)
    while cur.size:
        levels.append(cur)
        nd = nodes[cur]
        k = _popc(nd["imask"])
        cur = np.concatenate([np.arange(b, b + c, dtype=np.int64) for b, c in zip(nd["child_base"].astype(np.int64), k) if c]) if k.any() else np.zeros(0, np.int64)
    return levels


def refit_nodes(pre_nodes, recs):
    """k_collapse's quantisation (kz_lbvh.cuh) of the exact box of every used slot, in the frame of their union; topology kept"""
    out = pre_nodes.copy()
    n = len(pre_nodes)
    rlo = np.fmin(np.fmin(recs[:, 0, :3], recs[:, 1, :3]), recs[:, 2, :3])
    rhi = np.fmax(np.fmax(recs[:, 0, :3], recs[:, 1, :3]), recs[:, 2, :3])
    blo = np.zeros((n, 3), np.float32); bhi = np.zeros((n, 3), np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        for idx in reversed(node_levels(pre_nodes)):
            nd = pre_nodes[idx]
            m = len(idx)
            slo = np.full((m, 8, 3), np.inf, np.float32); shi = np.full((m, 8, 3), -np.inf, np.float32)
            used = np.zeros((m, 8), bool)
            imask = nd["imask"].astype(np.uint32); trimask = nd["trimask"].astype(np.uint32)
            for s in range(8):
                inner = ((imask >> s) & 1).astype(bool)
                ch = nd["child_base"].astype(np.int64) + _popc(imask & np.uint32((1 << s) - 1))
                slo[inner, s] = blo[ch[inner]]; shi[inner, s] = bhi[ch[inner]]
                bits = (trimask >> np.uint32(3 * s)) & np.uint32(7)
                for k in range(3):
                    has = ((bits >> np.uint32(k)) & 1).astype(bool) & ~inner
                    t = nd["tri_base"].astype(np.int64) + _popc(trimask & np.uint32((1 << (3 * s + k)) - 1))
                    slo[has, s] = np.fmin(slo[has, s], rlo[t[has]]); shi[has, s] = np.fmax(shi[has, s], rhi[t[has]])
                used[:, s] = inner | (bits != 0)
            nlo = slo.min(1); nhi = shi.max(1)
            blo[idx] = nlo; bhi[idx] = nhi
            out["p"][idx] = nlo + np.float32(0.0)
            ext = nhi.astype(np.float64) - nlo.astype(np.float64)
            ee = np.where(ext > 0, np.frexp(np.where(ext > 0, ext, 1.0) / 255.0)[1], -126)
            biased = np.clip(ee + 127, 1, 254)
            while True:
                up = (biased < 254) & (np.ceil(ext / np.ldexp(1.0, biased - 127)) > 255.0)
                if not up.any():
                    break
                biased = biased + up
            out["e"][idx] = biased.astype(np.uint8)
            sc = np.ldexp(1.0, biased - 127)[:, None, :]
            qlo = np.clip(np.floor((slo.astype(np.float64) - nlo[:, None, :].astype(np.float64)) / sc), 0, 255)
            qhi = np.clip(np.ceil((shi.astype(np.float64) - nlo[:, None, :].astype(np.float64)) / sc), 0, 255)
            u = used[:, None, :]
            out["qlo"][idx] = np.where(u, np.nan_to_num(qlo).astype(np.uint8).transpose(0, 2, 1), nd["qlo"])
            out["qhi"][idx] = np.where(u, np.nan_to_num(qhi).astype(np.uint8).transpose(0, 2, 1), nd["qhi"])
    return out


def check_rule(pre_nodes, pre_tris, post_nodes, post_tris, d):
    recs = refit_records(pre_tris, d)
    assert post_tris.tobytes() == recs.tobytes()
    for f in TOPOLOGY:
        assert np.array_equal(post_nodes[f], pre_nodes[f]), f
    want = refit_nodes(pre_nodes, recs)
    bad = np.nonzero(want.view(np.uint8).reshape(-1, 80) != post_nodes.view(np.uint8).reshape(-1, 80))[0]
    assert bad.size == 0, f"{np.unique(bad).size} of {len(want)} nodes differ, first {bad[0]}: want {want[bad[0]]} got {post_nodes[bad[0]]}"


def _occluded_pair(O, X, rays):
    rr = rays.copy()
    rr["tmax"] = np.where(np.isinf(rr["tmax"]), np.float32(50.0), rr["tmax"])
    return O.occluded(rr, 1e-3), X.occluded(rr, 1e-3)


# ------------------------------------------------------------------------------------------------------------ CPU (host emulation)
@pytest.mark.parametrize("motion", MOTIONS)
@pytest.mark.parametrize("name", sorted(SCENES))
def test_refit_emu_matches_oracle(kzo, emu, name, motion):
    import refit_emu
    sb = SCENES[name]()
    d = sb.desc()
    E = refit_emu.RefitEmu(d)
    pre_nodes, pre_tris = E.accel_dump()
    pre_nodes = pre_nodes.view(NODE_DTYPE).reshape(-1)
    keep = []
    dd = moved(d, deform(d, motion), keep)
    E.refit(dd)
    post_nodes, post_tris = E.accel_dump()
    check_rule(pre_nodes, pre_tris, post_nodes.view(NODE_DTYPE).reshape(-1), post_tris, dd)
    used = np.concatenate([_positions(dd, g)[_indices(dd, g)].reshape(-1, 3) for g in range(dd.n_meshes)])
    assert E.scene_max_abs() == float(np.abs(used).max())
    O = kzo.Oracle(dd)
    rays = np.concatenate([E.camera_rays(np.c_[np.random.default_rng(4).uniform(0, 1, (4096, 2)) * [dd.camera.width, dd.camera.height],
                                               np.full((4096, 2), 0.5)].astype(np.float32)), probe_rays(dd)])
    ho = O.trace(rays)
    assert E.trace(rays).tobytes() == ho.tobytes()
    assert (ho["geom_id"] != INVALID).mean() > 0.05
    (oo, so), (oe, se) = _occluded_pair(O, E, rays)
    assert np.array_equal(oo, oe) and np.array_equal(so, se)
    rr = rays.copy(); rr["tmax"] = np.where(np.isinf(rr["tmax"]), np.float32(50.0), rr["tmax"])
    oe, se, _ = E.occluded_early(rr, 1e-3)                 # the device's walk: stops early outside the invisible emitters' bounds
    assert np.array_equal(oo, oe) and np.array_equal(so, se)
    E.close(); O.close()


@pytest.mark.parametrize("name", ["cornell", "studio"])
def test_refit_emu_moved_emitters_walk(kzo, emu, name):
    """emitters moved (an invisible one into the way of shadow rays): the walk with the early stop (bounds of the invisible emitters)
    and the plain closest-hit walk both answer as the oracle"""
    import refit_emu
    sb = SCENES[name]()
    d = sb.desc()
    E = refit_emu.RefitEmu(d)
    lights = [g for g in range(d.n_meshes) if d.meshes[g].light >= 0]
    g = lights[-1]
    P = _positions(d, g)
    keep = []
    dd = moved(d, {g: (P - P.mean(0) + np.array([0.1, -0.2, 0.0], np.float32)).astype(np.float32)}, keep)     # into the middle of the scene
    E.refit(dd)
    O = kzo.Oracle(dd)
    rays = probe_rays(dd, 20000, seed=8)
    rays["tmax"] = np.where(np.isinf(rays["tmax"]), np.float32(30.0), rays["tmax"])
    oo, so = O.occluded(rays, 1e-3)
    oe, se, _ = E.occluded_early(rays, 1e-3)
    assert np.array_equal(oo, oe) and np.array_equal(so, se)
    assert so.max() >= 2
    E.close(); O.close()


# ------------------------------------------------------------------------------------------------------------ GPU
IMAGE_RELMSE_TOL = 2e-4          # as test_gpu_parity: GPU vs oracle at equal samples


def _update(G, d, dd, positions):
    for g in sorted(positions):
        G.mesh_update(g, _positions(dd, g))


def _dump(G, device=0):
    nodes, tris = G.accel_dump(device)
    return nodes.view(NODE_DTYPE).reshape(-1), tris


def _gpu_rays(dd):
    rng = np.random.default_rng(4)
    s4 = np.c_[rng.uniform(0, 1, (4096, 2)) * [dd.camera.width, dd.camera.height], np.full((4096, 2), 0.5)].astype(np.float32)
    return s4, probe_rays(dd)


@pytest.mark.gpu
@pytest.mark.parametrize("builder", [pk.BUILD_HOST_SAH, pk.BUILD_LBVH])
@pytest.mark.parametrize("name", sorted(SCENES))
def test_refit_gpu_exact_hits_and_node_bytes(kzo, gpu_lib, name, builder):
    """after mesh_update + refit: trace equals the oracle on the moved scene and a fresh upload + build, bit for bit; occluded equals the
    oracle; the refitted nodes and records equal the numpy restatement applied to the pre-refit topology"""
    sb = SCENES[name]()
    d = sb.desc()
    for motion in MOTIONS:
        keep = []
        pos = deform(d, motion)
        dd = moved(d, pos, keep)
        G = pk.Gpu(d, builder=builder)
        _update(G, d, dd, pos)
        pre_nodes, pre_tris = _dump(G)                   # the topology of the build, boxes of the old positions
        G.refit()
        post_nodes, post_tris = _dump(G)
        check_rule(pre_nodes, pre_tris, post_nodes, post_tris, dd)
        O, F = kzo.Oracle(dd), pk.Gpu(dd, builder=builder)
        s4, probe = _gpu_rays(dd)
        rays = np.concatenate([O.camera_rays(s4), probe])
        ho = O.trace(rays)
        assert G.trace(rays).tobytes() == ho.tobytes(), motion
        assert F.trace(rays).tobytes() == ho.tobytes(), motion
        assert (ho["geom_id"] != INVALID).mean() > 0.05
        (oo, so), (og, sg) = _occluded_pair(O, G, rays)
        assert np.array_equal(oo, og) and np.array_equal(so, sg), motion
        G.close(); O.close(); F.close()


@pytest.mark.gpu
def test_refit_gpu_full_size_from_device_tensor(kzo, gpu_lib):
    """a 10^7-triangle LBVH soup moved on the device with torch and updated from the tensor's pointer: 2^18 primary + 2^18 incoherent
    rays against the oracle on the moved soup (as test_full_size_sampled_oracle)"""
    torch = pytest.importorskip("torch")
    n = 10_000_000
    sb = scenes.soup_scene(n)
    d = sb.desc()
    G = pk.Gpu(d, builder=pk.BUILD_LBVH)
    P = torch.from_numpy(_positions(d, 0)).cuda()
    edge = 2.0 * n ** (-1.0 / 3.0)
    g = torch.Generator(device="cuda").manual_seed(11)
    P += (torch.randn(P.shape, device="cuda", generator=g) * (0.5 * edge)).to(torch.float32)
    torch.cuda.synchronize()
    G.mesh_update(0, P.data_ptr())
    G.refit()
    keep = []
    dd = moved(d, {0: P.cpu().numpy()}, keep)
    del P
    O = kzo.Oracle(dd)
    rays = np.concatenate([scenes.primary_rays(512), scenes.incoherent_rays(1 << 18)])
    a, b = O.trace(rays), G.trace(rays)
    assert a.tobytes() == b.tobytes()
    assert 0.5 < (a["geom_id"] != INVALID).mean() < 1.0
    occ_o, seg_o = O.occluded(rays[-(1 << 16):], 1e-4)
    occ_g, seg_g = G.occluded(rays[-(1 << 16):], 1e-4)
    assert np.array_equal(occ_o, occ_g) and np.array_equal(seg_o, seg_g)
    O.close(); G.close()


def _cornell_two_kinds_of_lights():
    sb = scenes.cornell_scene(48, 48, 16)
    sb.lights[0].primary_visibility = 1                 # the ceiling light is seen by the camera, the small one is not
    return sb


@pytest.mark.gpu
def test_refit_gpu_moved_emitters(kzo, gpu_lib):
    """moved visible and invisible emitters sample as a fresh upload of the moved scene (area CDF, normalisation, bounds of the invisible
    ones); an invisible emitter moved into the shadow rays' way is stepped through as the oracle steps through it"""
    sb = _cornell_two_kinds_of_lights()
    d = sb.desc()
    lights = [g for g in range(d.n_meshes) if d.meshes[g].light >= 0]
    assert len(lights) == 2
    vis, inv = lights
    Pv, Pi = _positions(d, vis), _positions(d, inv)
    R = np.array([[0.8, 0.0, 0.6], [0.0, 1.0, 0.0], [-0.6, 0.0, 0.8]], np.float32)
    pos = {vis: ((Pv - Pv.mean(0)) @ R.T * np.float32(1.3) + Pv.mean(0) + np.array([0.2, -0.05, 0.1], np.float32)).astype(np.float32),
           inv: (Pi - Pi.mean(0) + np.array([0.05, -0.1, -0.1], np.float32)).astype(np.float32)}          # to the middle of the box
    keep = []
    dd = moved(d, pos, keep)
    G, F, O = pk.Gpu(d), pk.Gpu(dd), kzo.Oracle(dd)
    _update(G, d, dd, pos)
    G.refit()
    rng = np.random.default_rng(9)
    ref = rng.uniform(-0.95, 0.95, (20000, 3)).astype(np.float32)
    u5 = rng.uniform(0, 1, (20000, 5)).astype(np.float32)
    assert G.light_sample_dump(ref, u5).tobytes() == F.light_sample_dump(ref, u5).tobytes()
    rays = scenes.incoherent_rays(100000, extent=0.95)
    rays["tmax"] *= 1.5
    (oo, so), (og, sg) = O.occluded(rays, 1e-3), G.occluded(rays, 1e-3)
    assert np.array_equal(oo, og) and np.array_equal(so, sg)
    assert sg.max() >= 2
    G.close(); F.close(); O.close()


def _render_pair(G, F):
    G.stats(reset=True); fg = G.render(); sg = G.stats(reset=True)
    F.stats(reset=True); ff = F.render(); sf = F.stats(reset=True)
    for key in ("paths", "rays_extension", "rays_shadow", "vertices"):
        assert sg[key] == sf[key], key
    np.testing.assert_allclose(fg, ff, rtol=1e-4, atol=1e-5)
    return fg, sg


@pytest.mark.gpu
@pytest.mark.parametrize("hint", [0, 2])
def test_refit_gpu_render_moved_sphere_and_light(kzo, gpu_lib, hint):
    """Cornell with the sphere and a light moved: the frame is held to the oracle's; against a fresh upload + build the same paths with
    the same counts and frames equal to the atomic splats' rounding; with primary-hit hints carried across the refit, they are used"""
    sb = _cornell_two_kinds_of_lights()
    d = sb.desc()
    sphere = max((g for g in range(d.n_meshes) if d.meshes[g].normals), key=lambda g: d.meshes[g].n_triangles)
    light = [g for g in range(d.n_meshes) if d.meshes[g].light >= 0][0]
    pos = {sphere: _positions(d, sphere) + np.array([0.5, 0.1, -0.3], np.float32), light: _positions(d, light) + np.array([0.25, -0.02, 0.1], np.float32)}
    keep = []
    dd = moved(d, pos, keep)
    for builder in (pk.BUILD_HOST_SAH, pk.BUILD_LBVH):
        G, F = pk.Gpu(d, builder=builder), pk.Gpu(dd, builder=builder)
        G.configure("primary_hint", hint); F.configure("primary_hint", hint)
        G.render()                                        # leaves hints of the old frame behind
        _update(G, d, dd, pos)
        with pytest.raises(RuntimeError, match="kzgpu_accel_refit"):
            G.render()
        G.refit()
        fg, sg = _render_pair(G, F)
        assert (sg["rays_seeded"] > 0) == (hint == 2)
        if builder == pk.BUILD_HOST_SAH:
            O = kzo.Oracle(dd)
            ro, _ = O.resolve(O.render()); rg, _ = G.resolve(fg)
            assert scenes.rel_mse(rg, ro).max() < IMAGE_RELMSE_TOL
            O.close()
        G.close(); F.close()


def _studio_camera(sb, x):
    c2w = np.array(sb.camera.camera_to_world, np.float32).reshape(4, 4).copy()
    c2w[0, 3] += x; c2w[2, 3] += 0.4 * x
    return c2w


@pytest.mark.gpu
def test_refit_gpu_camera_update(kzo, gpu_lib):
    """camera_update: camera rays equal a fresh upload's bit for bit (the oracle's to its tolerance), the studio frame after a camera
    move is held to the oracle's and to a fresh upload's; another film size is rejected"""
    sb = scenes.studio_scene(96, 64, 16)
    d = sb.desc()
    G = pk.Gpu(d)
    G.configure("primary_hint", 2)
    G.render()
    c2w = _studio_camera(sb, 0.7)
    G.camera_update(96, 64, 49.13434207760448, c2w, near=0.10000000149011612, far=100.0)
    sb2 = scenes.studio_scene(96, 64, 16)
    sb2.set_camera(96, 64, 49.13434207760448, c2w, near=0.10000000149011612, far=100.0)
    d2 = sb2.desc()
    F, O = pk.Gpu(d2), kzo.Oracle(d2)
    F.configure("primary_hint", 2)
    rng = np.random.default_rng(2)
    s4 = rng.uniform(0, 1, (5000, 4)).astype(np.float32) * np.array([96, 64, 1, 1], np.float32)
    a, b = G.camera_rays(s4), F.camera_rays(s4)
    assert a.tobytes() == b.tobytes()
    c = O.camera_rays(s4)
    for k in ("o", "d", "tmin", "tmax"):
        assert np.allclose(c[k], a[k], rtol=4e-6, atol=2e-7)
    fg, sg = _render_pair(G, F)
    assert sg["rays_seeded"] > 0
    ro, _ = O.resolve(O.render()); rg, _ = G.resolve(fg)
    assert scenes.rel_mse(rg, ro).max() < IMAGE_RELMSE_TOL
    for w, h in ((97, 64), (96, 63)):
        with pytest.raises(RuntimeError, match=r"camera_update failed \(-1\)"):
            G.camera_update(w, h, 49.0, c2w)
    assert G.camera_rays(s4).tobytes() == b.tobytes()
    G.close(); F.close(); O.close()


@pytest.mark.gpu
def test_refit_gpu_state_and_validation(gpu_lib):
    """call order (KZ_ERR_STATE) and argument checks (KZ_ERR_INVALID, the scene unchanged afterwards); update -> accel_build equals a
    fresh upload"""
    sb = scenes.cornell_scene(16, 16, 4)
    d = sb.desc()
    lib = C.CDLL(gpu_lib)
    lib.kzgpu_last_error.restype = C.c_char_p
    h = C.c_void_p()
    assert lib.kzgpu_create(None, 0, C.byref(h)) == 0
    P0 = _positions(d, 0)
    f32 = lambda a: a.ctypes.data_as(pk.c_float_p)
    assert lib.kzgpu_mesh_update(h, 0, f32(P0), None) == -4                 # nothing uploaded
    assert lib.kzgpu_scene_upload(h, C.byref(d)) == 0
    assert lib.kzgpu_accel_refit(h) == -4                                   # nothing built
    assert lib.kzgpu_accel_build(h, 0) == 0
    rays = probe_rays(d, 5000)
    ref = np.zeros(len(rays), pk.HIT_DTYPE)
    assert lib.kzgpu_trace(h, 0, rays.ctypes.data_as(C.c_void_p), C.c_size_t(len(rays)), 0, ref.ctypes.data_as(C.c_void_p)) == 0
    sphere = [g for g in range(d.n_meshes) if d.meshes[g].normals][0]
    Ps = _positions(d, sphere) + np.float32(0.3)
    nrm = np.zeros_like(P0)
    for args in ((d.n_meshes, f32(Ps), None), (-1, f32(Ps), None), (0, None, None), (0, f32(P0 + 1), f32(nrm))):
        assert lib.kzgpu_mesh_update(h, *args) == -1
        hits = np.zeros(len(rays), pk.HIT_DTYPE)                            # rejected: the scene and the accel are as they were
        assert lib.kzgpu_trace(h, 0, rays.ctypes.data_as(C.c_void_p), C.c_size_t(len(rays)), 0, hits.ctypes.data_as(C.c_void_p)) == 0
        assert hits.tobytes() == ref.tobytes()
    assert lib.kzgpu_camera_update(h, None) == -1
    assert lib.kzgpu_mesh_update(h, sphere, f32(Ps), f32(_positions(d, sphere) * 0 + np.float32(0.577))) == 0     # a mesh with normals takes them
    hits = np.zeros(len(rays), pk.HIT_DTYPE)
    assert lib.kzgpu_trace(h, 0, rays.ctypes.data_as(C.c_void_p), C.c_size_t(len(rays)), 0, hits.ctypes.data_as(C.c_void_p)) == -4
    assert b"kzgpu_accel_refit" in lib.kzgpu_last_error(h)
    frame = np.zeros((20, 20, 4), np.float32)
    req = pk.RenderReq(0, 0, 16, 16, 0, 4, 1)
    assert lib.kzgpu_render(h, C.byref(req), f32(frame)) == -4
    # update -> build (instead of refit) is a fresh upload's accel
    assert lib.kzgpu_accel_build(h, 1) == 0
    keep = []
    dd = moved(d, {sphere: Ps}, keep)
    F = pk.Gpu(dd, builder=pk.BUILD_LBVH)
    assert lib.kzgpu_trace(h, 0, rays.ctypes.data_as(C.c_void_p), C.c_size_t(len(rays)), 0, hits.ctypes.data_as(C.c_void_p)) == 0
    assert hits.tobytes() == F.trace(rays).tobytes()
    F.close()
    lib.kzgpu_destroy(h)


@pytest.mark.gpu
def test_refit_gpu_multi_device(kzo, gpu_lib):
    """every device refits its own copy: identical accel bytes everywhere, the last device traces as device 0 and the oracle"""
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    sb = scenes.cornell_scene(32, 32, 4)
    d = sb.desc()
    pos = deform(d, "jitter")
    keep = []
    dd = moved(d, pos, keep)
    for builder in (pk.BUILD_HOST_SAH, pk.BUILD_LBVH):
        G = pk.Gpu(d, devices=tuple(range(n)), builder=builder)
        _update(G, d, dd, pos)
        G.refit()
        n0, t0 = G.accel_dump(0)
        for g in range(1, n):
            ng, tg = G.accel_dump(g)
            assert ng.tobytes() == n0.tobytes() and tg.tobytes() == t0.tobytes()
        O = kzo.Oracle(dd)
        rays = probe_rays(dd, 20000)
        ho = O.trace(rays)
        assert G.trace(rays, device=n - 1).tobytes() == ho.tobytes() == G.trace(rays, device=0).tobytes()
        G.close(); O.close()
