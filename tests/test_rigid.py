"""Rigid motion: kzgpu_mesh_transform (kz_transform.h, k_transform_vertices) and the KZ_BUILD_LBVH_MESHES builder (kz_lbvh.cuh).

A transformed mesh must equal, bit for bit, the same arrays placed on the host the way the C++ host's OBJ loader applies `toWorld`
(Transform::point / Transform::normal, then the loader's normalisation); `place` below restates that in numpy float32, one rounding per
operation.  The per-mesh builder must keep every mesh in its own subtrees, lay its nodes out level by level (so a refit runs on it), and
-- like every accel -- give exactly the hits of the oracle, before and after transform + refit."""
import collections
import ctypes as C
import os

import numpy as np
import pytest

import scenes
import pykazen as pk
from test_refit import NODE_DTYPE, check_rule, refit_records, probe_rays, _positions, _indices, _popc, _occluded_pair

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INVALID = 0xFFFFFFFF
IMAGE_RELMSE_TOL = 2e-4          # as test_refit_gpu_render_moved_sphere_and_light
f32 = np.float32


# ------------------------------------------------------------------------------------------------------------ the arithmetic, in numpy
def place_points(M, P):
    """Transform::point (host/src/core.cpp:53-60): each row ((M0 x + M1 y) + M2 z) + M3, then divided by w"""
    M = np.asarray(M, f32).reshape(4, 4); P = np.asarray(P, f32).reshape(-1, 3)
    r = [((M[i, 0] * P[:, 0] + M[i, 1] * P[:, 1]) + M[i, 2] * P[:, 2]) + M[i, 3] for i in range(4)]
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        return np.stack([r[0] / r[3], r[1] / r[3], r[2] / r[3]], 1).astype(f32)


def place_normals(I, N):
    """Transform::normal (core.cpp:65-68), then the OBJ loader's normalisation (plugins.cpp:533-535)"""
    I = np.asarray(I, f32).reshape(4, 4); N = np.asarray(N, f32).reshape(-1, 3)
    r = np.stack([(I[0, j] * N[:, 0] + I[1, j] * N[:, 1]) + I[2, j] * N[:, 2] for j in range(3)], 1).astype(f32)
    z = r[:, 0] * r[:, 0] + (r[:, 1] * r[:, 1] + r[:, 2] * r[:, 2])
    pos = z > 0
    l = np.sqrt(np.where(pos, z, f32(1)))
    return np.where(pos[:, None], r / l[:, None], r).astype(f32)


def inverse(M):
    return np.linalg.inv(np.asarray(M, np.float64)).astype(f32)


def about(centre, A, t=(0, 0, 0)):
    """the float32 4x4 of p -> A (p - centre) + centre + t, composed in float64"""
    M = np.eye(4)
    M[:3, :3] = A
    M[:3, 3] = np.asarray(centre, np.float64) - np.asarray(A, np.float64) @ np.asarray(centre, np.float64) + np.asarray(t, np.float64)
    return M.astype(f32)


def rotation(axis, deg):
    a = np.asarray(axis, np.float64); a /= np.linalg.norm(a)
    th = np.radians(deg)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * K @ K


def _bits(a):
    return np.ascontiguousarray(a, f32).view(np.uint32)


# ------------------------------------------------------------------------------------------------------------ CPU
def _matrices():
    rng = np.random.default_rng(21)
    out = {}
    for k in range(4):
        out[f"affine{k}"] = about(rng.uniform(-1, 1, 3), rotation(rng.normal(size=3), rng.uniform(0, 180)) * rng.uniform(0.2, 3.0), rng.uniform(-5, 5, 3))
    P = about((0.1, 0.2, 0.3), rotation((1, 2, 3), 33), (1, -2, 0.5))
    P[3] = [0.05, -0.03, 0.02, 1.25]                                          # projective row: w != 1
    out["projective"] = P
    out["mirror"] = about((0.3, 0, 0), np.diag([-1.0, 1.0, 1.0]) @ rotation((0, 1, 0), 20), (0.2, 0.1, 0))
    out["scale1e3"] = about((0.1, -0.1, 0.2), 1000.0 * rotation((1, 1, 0), 10))
    return out


def test_transform_body_matches_numpy_restatement():
    """kz_transform.h compiled for the host equals the numpy restatement bit for bit: random affine matrices, a projective row, a
    mirror, a 10^3 scale; random normals, a zero normal and normals that are zero after the transform"""
    import transform_emu
    rng = np.random.default_rng(5)
    P = rng.uniform(-2, 2, (4096, 3)).astype(f32)
    N = rng.normal(size=(4096, 3)).astype(f32)
    N[0] = 0.0
    for name, M in _matrices().items():
        I = inverse(M)
        gp, gn = transform_emu.transform(M, I, P, N)
        assert np.array_equal(_bits(gp), _bits(place_points(M, P))), name
        assert np.array_equal(_bits(gn), _bits(place_normals(I, N))), name
        assert not np.any(gn[0])
    # an inverse whose upper 3x3 maps some normals to zero
    I = np.diag([1.0, 1.0, 0.0, 1.0]).astype(f32)
    Nz = np.array([[0, 0, 1], [0, 0, -2.5], [1, 0, 1]], f32)
    gp, gn = transform_emu.transform(np.eye(4, dtype=f32), I, Nz, Nz)
    assert np.array_equal(_bits(gn), _bits(place_normals(I, Nz)))
    assert not np.any(gn[:2]) and gn[2].tolist() == [1.0, 0.0, 0.0]
    assert np.array_equal(_bits(gp), _bits(Nz))


def _load_obj(tmp_path, obj, matrix=None):
    xml = tmp_path / ("m.xml" if matrix is None else "t.xml")
    tw = "" if matrix is None else ('<transform name="toWorld"><matrix value="' + " ".join("%.9g" % v for v in np.asarray(matrix, f32).reshape(-1)) +
                                    '"/></transform>')
    xml.write_text(f"""<?xml version="1.0" ?>
<scene>
    <integrator type="path_mis"/>
    <sampler type="independent"><integer name="sampleCount" value="1"/></sampler>
    <camera type="perspective"><integer name="width" value="8"/><integer name="height" value="8"/></camera>
    <mesh type="obj"><string name="filename" value="{obj}"/>{tw}<bsdf type="diffuse"/></mesh>
</scene>""")
    hs = pk.HostScene(str(xml))
    m = hs.desc.meshes[0]
    V = np.ctypeslib.as_array(m.positions, (m.n_vertices * 3,)).reshape(-1, 3).copy()
    hs.close()
    return V


@pytest.mark.parametrize("obj", ["tri_full.obj", "quads.obj", "dedup.obj"])
def test_host_loader_to_world_matches_restatement(tmp_path, obj):
    """the C++ host's OBJ loader with a non-trivial toWorld produces the restatement applied to the identity-loaded positions: the
    device's arithmetic is the host's"""
    import subprocess
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "nano-kazen_b200", "host")])
    path = os.path.join(ROOT, "tests", "golden", "obj", obj)
    V0 = _load_obj(tmp_path, path)
    for name, M in _matrices().items():
        M = np.where(M == 0, f32(0), M).astype(f32)                 # no -0 entries: the parser composes the matrix with the identity
        V = _load_obj(tmp_path, path, M)
        assert np.array_equal(_bits(V), _bits(place_points(M, V0))), name


# ------------------------------------------------------------------------------------------------------------ scenes
def multi_soup(k=27, n=1 << 12, grid=3, seed=7, size=96, spp=8):
    """k hash-soup clusters as separate meshes, one per cell of a grid x grid x grid lattice over [-1, 1]^3, under an environment light"""
    sb = pk.SceneBuilder()
    bs = sb.bsdf_diffuse((0.6, 0.5, 0.4))
    cell = 2.0 / grid
    for c in range(k):
        i, j, l = c % grid, (c // grid) % grid, c // (grid * grid)
        centre = np.array([-1 + cell * (i + 0.5), -1 + cell * (j + 0.5), -1 + cell * (l + 0.5)], f32)
        P = (scenes.hash_soup_numpy(n, seed=seed + c) * f32(0.4 * cell) + centre).astype(f32)
        sb.mesh(P, np.arange(3 * n, dtype=np.uint32).reshape(-1, 3), bs)
    sb.background = sb.tex_background(1.0, sb.tex_constant((0.8, 0.9, 1.0)))
    sb.set_camera(size, size, 40.0, pk.lookat((0.3, 0.4, -3.5), (0, 0, 0), (0, 1, 0)))
    sb.set_sampler("stratified", spp)
    sb.set_integrator(max_depth=4)
    return sb


SCENES = {
    "cornell": lambda: scenes.cornell_scene(32, 32, 4),
    "studio": lambda: scenes.studio_scene(48, 48, 4),
    "multi": multi_soup,
}


def _normals(d, g):
    m = d.meshes[g]
    return np.ctypeslib.as_array(m.normals, shape=(m.n_vertices * 3,)).reshape(-1, 3).copy() if m.normals else None


def placed(d, arrays, keep):
    """a copy of scene desc `d` whose meshes g in `arrays` have the given (positions, normals or None)"""
    dd = pk.SceneDesc.from_buffer_copy(d)
    meshes = (pk.MeshDesc * max(1, d.n_meshes))()
    for g in range(d.n_meshes):
        C.memmove(C.byref(meshes[g]), C.byref(d.meshes[g]), C.sizeof(pk.MeshDesc))
        if g in arrays:
            P, N = arrays[g]
            P = np.ascontiguousarray(P, f32); keep.append(P)
            meshes[g].positions = P.ctypes.data_as(pk.c_float_p)
            if N is not None:
                N = np.ascontiguousarray(N, f32); keep.append(N)
                meshes[g].normals = N.ctypes.data_as(pk.c_float_p)
    dd.meshes = meshes
    keep += [meshes, dd]
    return dd


def motion(d, kind, g):
    """the float32 matrix of one rigid motion of mesh g"""
    P = _positions(d, g)
    all_p = np.concatenate([_positions(d, k) for k in range(d.n_meshes)])
    size = float(np.abs(all_p).max())
    c = P.mean(0).astype(np.float64)
    if kind == "translate":
        return about(c, np.eye(3), np.array([7.0, -4.0, 5.0]) * size)
    if kind == "rotate":
        return about(c, rotation((1, 2, -1), 40 + 7 * g), (0.05, -0.02, 0.03))
    if kind == "mirror":
        return about(c, np.diag([1.0, -1.0, 1.0]) @ rotation((0, 0, 1), 15), (0.02, 0, 0))
    if kind == "scale":
        return about(c, 1000.0 * rotation((0, 1, 0), 5))
    raise ValueError(kind)


def apply(G, d, mats):
    """mesh_transform every (mesh, matrix) of `mats` on G; returns {mesh: (placed positions, placed normals)} in numpy"""
    out = {}
    for g, M in mats.items():
        I = inverse(M)
        G.mesh_transform(g, M, I)
        N = _normals(d, g)
        out[g] = (place_points(M, _positions(d, g)), None if N is None else place_normals(I, N))
    return out


def _dump(G, device=0):
    nodes, tris = G.accel_dump(device)
    return nodes.view(NODE_DTYPE).reshape(-1), tris


def check_mesh_subtrees(nodes, tris, d):
    """every slot of every node: its subtree holds triangles of one mesh, or every mesh it touches entirely"""
    total = collections.Counter({g: d.meshes[g].n_triangles for g in range(d.n_meshes)})
    geom = tris[:, 0, 3].view(np.uint32)
    below = {}                                             # node -> Counter of its subtree
    levels = []
    cur = [0] if len(nodes) else []
    while cur:
        levels.append(cur)
        cur = [int(nodes[i]["child_base"]) + k for i in cur for k in range(int(_popc(nodes[i]["imask"])))]
    checked = 0
    for lvl in reversed(levels):
        for i in lvl:
            nd = nodes[i]
            mine = collections.Counter()
            for s in range(8):
                if (int(nd["imask"]) >> s) & 1:
                    slot = below[int(nd["child_base"]) + int(_popc(int(nd["imask"]) & ((1 << s) - 1)))]
                else:
                    bits = (int(nd["trimask"]) >> (3 * s)) & 7
                    if not bits:
                        continue
                    first = int(nd["tri_base"]) + int(_popc(int(nd["trimask"]) & ((1 << (3 * s)) - 1)))
                    slot = collections.Counter(geom[first: first + bin(bits).count("1")].tolist())
                    assert len(slot) == 1, f"leaf slot of node {i} holds meshes {sorted(slot)}"
                assert len(slot) == 1 or all(slot[g] == total[g] for g in slot), f"slot {s} of node {i} holds part of a mesh among others"
                mine += slot
                checked += 1
            below[i] = mine
    assert below[0] == +total
    return checked


def _runs(starts, counts):
    """concatenation of arange(s, s + c) over (starts, counts)"""
    starts = np.asarray(starts, np.int64); counts = np.asarray(counts, np.int64)
    if counts.sum() == 0:
        return np.zeros(0, np.int64)
    ends = np.cumsum(counts)
    return np.repeat(starts - (ends - counts), counts) + np.arange(ends[-1])


def canonical(nodes, tris):
    """an accel's bytes in tree order: the LBVH collapse hands out node and triangle positions with atomics, so two builds of one tree
    may store it in a different order.  Nodes level by level, each level in the order of its parents' slots, child_base / tri_base
    zeroed; the triangle records of every node's leaf slots in the same order."""
    nodes = np.asarray(nodes).view(NODE_DTYPE).reshape(-1)
    levels, cur = [], np.zeros(1 if len(nodes) else 0, np.int64)
    while cur.size:
        levels.append(cur)
        nd = nodes[cur]
        cur = _runs(nd["child_base"], _popc(nd["imask"]))
    nd = nodes[np.concatenate(levels)] if levels else nodes[:0]
    recs = np.asarray(tris).reshape(-1, 3, 4)[_runs(nd["tri_base"], _popc(nd["trimask"]))]
    nd = nd.copy()
    nd["child_base"] = 0; nd["tri_base"] = 0
    return nd.tobytes() + recs.tobytes()


# ------------------------------------------------------------------------------------------------------------ GPU: the builder
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1 << 15, 1 << 20])
def test_lbvh_meshes_on_one_mesh_is_the_lbvh_without_presplit(gpu_lib, monkeypatch, n):
    """with one mesh the rank is constant: the same tree as KZ_BUILD_LBVH with KZ_LBVH_PRESPLIT=0, node for node and record for record"""
    sb = scenes.soup_scene(n)
    d = sb.desc()
    A = pk.Gpu(d, builder=pk.BUILD_LBVH_MESHES)
    monkeypatch.setenv("KZ_LBVH_PRESPLIT", "0")
    B = pk.Gpu(d, builder=pk.BUILD_LBVH)
    na, ta = A.accel_dump(); nb, tb = B.accel_dump()
    assert len(na) == len(nb) and len(ta) == len(tb) == n
    assert canonical(na, ta) == canonical(nb, tb)
    A.close(); B.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SCENES))
def test_lbvh_meshes_invariant_refit_and_hits(kzo, gpu_lib, name):
    """the slot rule on every node; the level layout passes the refit's check and a refit without motion leaves the bytes as built; trace
    and both shadow walks equal the oracle's"""
    sb = SCENES[name]()
    d = sb.desc()
    G = pk.Gpu(d, builder=pk.BUILD_LBVH_MESHES)
    nodes, tris = _dump(G)
    assert check_mesh_subtrees(nodes, tris, d) > d.n_meshes
    G.refit()
    n2, t2 = _dump(G)
    assert n2.tobytes() == nodes.tobytes() and t2.tobytes() == tris.tobytes()
    O = kzo.Oracle(d)
    rays = probe_rays(d)
    ho = O.trace(rays)
    assert G.trace(rays).tobytes() == ho.tobytes()
    assert (ho["geom_id"] != INVALID).mean() > 0.05
    (oo, so), (og, sg) = _occluded_pair(O, G, rays)
    assert np.array_equal(oo, og) and np.array_equal(so, sg)
    G.close(); O.close()


# ------------------------------------------------------------------------------------------------------------ GPU: transform + refit
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SCENES))
def test_transform_refit_exact_hits_and_bytes(kzo, gpu_lib, name):
    """translate far, rotate, mirror and scale by 10^3, one mesh and all meshes: after mesh_transform + refit of a KZ_BUILD_LBVH_MESHES
    accel the triangle records and nodes follow the refit rule over the numpy-placed rest pose, trace and both shadow walks equal the
    oracle on the moved scene and a fresh upload of the moved arrays with either existing builder"""
    sb = SCENES[name]()
    d = sb.desc()
    big = max((g for g in range(d.n_meshes) if d.meshes[g].light < 0), key=lambda g: d.meshes[g].n_triangles)
    for kind in ("translate", "rotate", "mirror", "scale"):
        for which in ("one", "all"):
            mats = {g: motion(d, kind, g) for g in ([big] if which == "one" else range(d.n_meshes))}
            G = pk.Gpu(d, builder=pk.BUILD_LBVH_MESHES)
            arrays = apply(G, d, mats)
            pre_nodes, pre_tris = _dump(G)
            G.refit()
            keep = []
            dd = placed(d, arrays, keep)
            post_nodes, post_tris = _dump(G)
            check_rule(pre_nodes, pre_tris, post_nodes, post_tris, dd)
            O = kzo.Oracle(dd)
            rays = probe_rays(dd)
            ho = O.trace(rays)
            assert G.trace(rays).tobytes() == ho.tobytes(), (kind, which)
            F = pk.Gpu(dd, builder=pk.BUILD_LBVH if which == "one" else pk.BUILD_HOST_SAH)
            assert F.trace(rays).tobytes() == ho.tobytes(), (kind, which)
            assert (ho["geom_id"] != INVALID).mean() > 0.05
            (oo, so), (og, sg) = _occluded_pair(O, G, rays)
            assert np.array_equal(oo, og) and np.array_equal(so, sg), (kind, which)
            G.close(); O.close(); F.close()


@pytest.mark.gpu
def test_transform_vertex_bytes_rest_pose_and_update(gpu_lib):
    """intersection records (positions and normals) equal a context uploaded with the pre-placed arrays; a second transform applies to
    the rest pose, not to the first result; mesh_update then mesh_transform places the updated arrays"""
    sb = scenes.cornell_scene(32, 32, 4)
    d = sb.desc()
    sphere = max((g for g in range(d.n_meshes) if d.meshes[g].normals), key=lambda g: d.meshes[g].n_triangles)
    c = _positions(d, sphere).mean(0)
    M1 = about(c, rotation((0, 1, 1), 50) * 0.7, (0.1, 0.2, -0.1))
    M2 = about(c, np.diag([-1.0, 1.0, 1.0]) @ rotation((1, 0, 0), 25), (-0.2, 0.0, 0.1))
    G = pk.Gpu(d, builder=pk.BUILD_LBVH_MESHES)
    G.mesh_transform(sphere, M1, inverse(M1))
    G.mesh_transform(sphere, M2)                                    # inverse computed by pykazen: np.linalg.inv rounded to float32
    G.refit()
    keep = []
    want = {sphere: (place_points(M2, _positions(d, sphere)), place_normals(inverse(M2), _normals(d, sphere)))}
    dd = placed(d, want, keep)
    F = pk.Gpu(dd, builder=pk.BUILD_LBVH)
    P = want[sphere][0][_indices(d, sphere)]
    rng = np.random.default_rng(3)
    rays = np.zeros(20000, pk.RAY_DTYPE)                            # aimed at the placed sphere and all over the box
    w = rng.dirichlet((1, 1, 1), 10000)
    o = rng.uniform(-0.9, 0.9, (20000, 3)).astype(f32)
    aim = np.concatenate([(P[rng.integers(0, len(P), 10000)] * w[:, :, None]).sum(1) - o[:10000], rng.normal(size=(10000, 3))])
    rays["o"] = o; rays["d"] = (aim / np.linalg.norm(aim, axis=1, keepdims=True)).astype(f32)
    rays["tmin"] = f32(1e-4); rays["tmax"] = np.inf
    a, b = G.intersection_dump(rays), F.intersection_dump(rays)
    assert np.array_equal(_bits(a), _bits(b))
    assert (a[:, 1] == sphere).mean() > 0.3
    # mesh_update replaces the rest pose: the next transform places the updated arrays
    P2 = (_positions(d, sphere) * f32(0.8)).astype(f32)
    N2 = _normals(d, sphere)[::-1].copy()
    G.mesh_update(sphere, P2, N2)
    G.mesh_transform(sphere, M1, inverse(M1))
    G.refit()
    _, tris = G.accel_dump()
    keep = []
    dd = placed(d, {sphere: (place_points(M1, P2), place_normals(inverse(M1), N2))}, keep)
    assert tris.tobytes() == refit_records(tris, dd).tobytes()
    F.close()
    F = pk.Gpu(dd, builder=pk.BUILD_LBVH)
    assert np.array_equal(_bits(G.intersection_dump(rays)), _bits(F.intersection_dump(rays)))
    G.close(); F.close()


def _cornell_two_kinds_of_lights():
    sb = scenes.cornell_scene(48, 48, 16)
    sb.lights[0].primary_visibility = 1
    return sb


@pytest.mark.gpu
def test_transform_emitters(kzo, gpu_lib):
    """a rotated and translated area light samples as a freshly uploaded one, bit for bit; an invisible emitter moved into the shadow
    rays' way is stepped through as the oracle steps through it"""
    sb = _cornell_two_kinds_of_lights()
    d = sb.desc()
    vis, inv = [g for g in range(d.n_meshes) if d.meshes[g].light >= 0]
    cv, ci = _positions(d, vis).mean(0), _positions(d, inv).mean(0)
    mats = {vis: about(cv, rotation((1, 0, 1), 35) * 1.3, (0.2, -0.05, 0.1)),
            inv: about(ci, rotation((0, 1, 0), 60), (0.05, -0.1, -0.1) - ci)}          # to the middle of the box
    G = pk.Gpu(d)
    arrays = apply(G, d, mats)
    G.refit()
    keep = []
    dd = placed(d, arrays, keep)
    F, O = pk.Gpu(dd), kzo.Oracle(dd)
    rng = np.random.default_rng(9)
    ref = rng.uniform(-0.95, 0.95, (20000, 3)).astype(f32)
    u5 = rng.uniform(0, 1, (20000, 5)).astype(f32)
    assert G.light_sample_dump(ref, u5).tobytes() == F.light_sample_dump(ref, u5).tobytes()
    rays = scenes.incoherent_rays(100000, extent=0.95)
    rays["tmax"] *= 1.5
    (oo, so), (og, sg) = O.occluded(rays, 1e-3), G.occluded(rays, 1e-3)
    assert np.array_equal(oo, og) and np.array_equal(so, sg)
    assert sg.max() >= 2
    G.close(); F.close(); O.close()


@pytest.mark.gpu
def test_transform_state_and_validation(gpu_lib):
    """KZ_ERR_STATE before an upload and for trace between transform and refit; KZ_ERR_INVALID for a bad mesh index, a NULL matrix, a
    NULL inverse for a mesh with normals and non-finite entries, each changing nothing"""
    sb = scenes.cornell_scene(16, 16, 4)
    d = sb.desc()
    lib = C.CDLL(gpu_lib)
    lib.kzgpu_last_error.restype = C.c_char_p
    h = C.c_void_p()
    assert lib.kzgpu_create(None, 0, C.byref(h)) == 0
    fp = lambda a: a.ctypes.data_as(pk.c_float_p)
    M = about((0, 0, 0), rotation((0, 1, 0), 30), (0.1, 0, 0))
    I = inverse(M)
    assert lib.kzgpu_mesh_transform(h, 0, fp(M), fp(I)) == -4                       # nothing uploaded
    assert lib.kzgpu_scene_upload(h, C.byref(d)) == 0
    assert lib.kzgpu_accel_build(h, pk.BUILD_LBVH_MESHES) == 0
    rays = probe_rays(d, 5000)

    def trace():
        hits = np.zeros(len(rays), pk.HIT_DTYPE)
        rc = lib.kzgpu_trace(h, 0, rays.ctypes.data_as(C.c_void_p), C.c_size_t(len(rays)), 0, hits.ctypes.data_as(C.c_void_p))
        return rc, hits
    rc, ref = trace()
    assert rc == 0
    sphere = [g for g in range(d.n_meshes) if d.meshes[g].normals][0]
    nan, inf = M.copy(), I.copy()
    nan[1, 2] = np.nan; inf[0, 0] = np.inf
    for args in ((d.n_meshes, fp(M), fp(I)), (-1, fp(M), fp(I)), (0, None, fp(I)), (sphere, fp(M), None), (0, fp(nan), fp(I)), (sphere, fp(M), fp(inf))):
        assert lib.kzgpu_mesh_transform(h, *args) == -1
        rc, hits = trace()
        assert rc == 0 and hits.tobytes() == ref.tobytes()
    assert lib.kzgpu_mesh_transform(h, sphere, fp(M), fp(I)) == 0
    assert trace()[0] == -4
    assert b"kzgpu_accel_refit" in lib.kzgpu_last_error(h)
    assert lib.kzgpu_accel_refit(h) == 0
    rc, hits = trace()
    assert rc == 0 and hits.tobytes() != ref.tobytes()
    lib.kzgpu_destroy(h)


@pytest.mark.gpu
def test_scene_upload_drops_rest_copies(gpu_lib):
    """a transform keeps the rest pose in HBM (12 bytes per vertex); the next scene_upload releases it, and cycles of upload, transform
    and refit keep device free memory within the bound of test_ctx_lifetime"""
    torch = pytest.importorskip("torch")
    n = 1 << 22
    sb = scenes.soup_scene(n)
    d = sb.desc()
    G = pk.Gpu(d, builder=pk.BUILD_LBVH_MESHES)

    def free():
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        return torch.cuda.mem_get_info()[0]
    M = about((0, 0, 0), rotation((1, 1, 1), 20), (0.1, 0.2, 0.3))

    def cycle():
        G._call("scene_upload", G.h, C.byref(d))
        G._call("accel_build", G.h, C.c_int(pk.BUILD_LBVH_MESHES))
        G.mesh_transform(0, M)
        G.refit()
    cycle()
    held = free()
    G._call("scene_upload", G.h, C.byref(d))                         # drops the accel and the rest copy
    G._call("accel_build", G.h, C.c_int(pk.BUILD_LBVH_MESHES))
    rest = 3 * n * 12
    assert free() - held > 0.9 * rest
    before = free()
    for _ in range(3):
        cycle()
    G._call("scene_upload", G.h, C.byref(d))
    G._call("accel_build", G.h, C.c_int(pk.BUILD_LBVH_MESHES))
    assert before - free() < (64 << 20)
    G.close()


@pytest.mark.gpu
def test_transform_multi_device(kzo, gpu_lib):
    """every device places its own rest copy and refits its own accel: identical vertex and accel bytes everywhere"""
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    sb = multi_soup()
    d = sb.desc()
    G = pk.Gpu(d, devices=tuple(range(n)), builder=pk.BUILD_LBVH_MESHES)
    arrays = apply(G, d, {g: motion(d, "rotate", g) for g in range(0, d.n_meshes, 2)})
    G.refit()
    n0, t0 = G.accel_dump(0)
    rays = probe_rays(d, 20000)
    keep = []
    dd = placed(d, arrays, keep)
    O = kzo.Oracle(dd)
    ho = O.trace(rays)
    for g in range(n):
        ng, tg = G.accel_dump(g)
        assert ng.tobytes() == n0.tobytes() and tg.tobytes() == t0.tobytes()
        assert G.trace(rays, device=g).tobytes() == ho.tobytes()
    G.close(); O.close()


@pytest.mark.gpu
def test_transform_refit_render_matches_oracle(kzo, gpu_lib):
    """the multi-mesh scene rendered after transform + refit: the frame is held to the oracle's on the moved scene"""
    sb = multi_soup(size=48, spp=16)
    d = sb.desc()
    G = pk.Gpu(d, builder=pk.BUILD_LBVH_MESHES)
    G.render()
    arrays = apply(G, d, {g: motion(d, "rotate" if g % 2 else "mirror", g) for g in range(d.n_meshes)})
    G.refit()
    keep = []
    dd = placed(d, arrays, keep)
    O = kzo.Oracle(dd)
    rg, _ = G.resolve(G.render()); ro, _ = O.resolve(O.render())
    assert scenes.rel_mse(rg, ro).max() < IMAGE_RELMSE_TOL
    G.close(); O.close()
