"""The primary-hit seed split the way the device runs it: k_raygen runs the seed test on the ray it has just generated (kz_seed_hit) and
leaves the hit in the path's hit record, k_extend<true> installs it in the ray's fresh traversal (kz_trav_preset).  On the host emulation,
for every kind of hint, the hit kz_seed_hit returns must be the preset kz_trav_seed makes, bit for bit, and a traversal started from it
must return the same closest hit as an unseeded one."""
import numpy as np
import pytest

import scenes
from test_primary_hint import SCENES, INVALID, _camera_rays, _seeds


def _emu(desc):
    import raygen_seed_emu
    return raygen_seed_emu.RaygenSeedEmu(desc)


def _check(E, rays, ref, seeds):
    """kz_seed_hit == kz_trav_seed's preset, the preset is installed exactly when the seed test hit, and the traversal it starts returns
    the unseeded closest hit; returns the number of hints taken"""
    pure, trav, taken = E.seed_split(rays, seeds)
    assert set(np.unique(taken).tolist()) <= {0, 7}, np.unique(taken)
    on = taken == 7
    assert pure[on].tobytes() == trav[on].tobytes()
    # not taken: k_raygen's record stays the invalid hit, the traversal stays as kz_trav_init left it
    assert (pure["geom_id"][~on] == INVALID).all() and (pure["prim_id"][~on] == INVALID).all()
    assert (trav["geom_id"][~on] == INVALID).all() and (trav["prim_id"][~on] == INVALID).all()
    assert trav["t"][~on].tobytes() == rays["tmax"][~on].tobytes()
    assert E.trace_preset(rays, pure).tobytes() == ref.tobytes()
    return int(on.sum())


@pytest.mark.parametrize("name", sorted(SCENES))
def test_raygen_seed_matches_trav_seed(emu, name):
    sb = SCENES[name]()          # holds the arrays the descriptor points into
    d = sb.desc()
    E = _emu(d)
    rays = _camera_rays(E, d)
    ref = E.trace(rays)
    hit = ref["geom_id"] != INVALID
    n_tris = np.array([d.meshes[g].n_triangles for g in range(d.n_meshes)], np.int64)
    g = np.where(hit, ref["geom_id"], 0).astype(np.int64)
    p = np.where(hit, ref["prim_id"], 0).astype(np.int64)
    behind = rays.copy()
    behind["tmin"] = np.where(hit, np.nextafter(ref["t"], np.float32(np.inf)), behind["tmin"])
    second = E.trace(behind)

    assert _check(E, rays, ref, _seeds(ref["geom_id"], ref["prim_id"])) == int(hit.sum())                  # the right triangle
    _check(E, rays, ref, _seeds(np.roll(ref["geom_id"], 1), np.roll(ref["prim_id"], 1)))                     # the neighbouring sample's hit
    _check(E, rays, ref, _seeds(g, (p + 1) % n_tris[g]))                                                     # the neighbouring triangle
    k = _check(E, rays, ref, _seeds(second["geom_id"], second["prim_id"]))                                   # hit, but behind the closest
    if name != "cornell":
        assert k > 0
    _check(E, rays, ref, _seeds(ref["geom_id"][::-1], ref["prim_id"][::-1]))                                 # mostly missed
    nm = d.n_meshes
    for gg, pp in ((nm, 0), (INVALID, 0), (0, int(n_tris[0])), (0, INVALID), (INVALID, INVALID)):          # out of range
        assert _check(E, rays, ref, _seeds(np.full(len(rays), gg), np.full(len(rays), pp))) == 0
    # NaN rays (k_raygen's padding lanes are NaN rays) never take a seed, not even the triangle the ray would hit without the NaN
    nan = rays.copy()
    for k, (field, axis) in enumerate((("o", 0), ("o", 2), ("d", 1), ("d", 2), ("tmin", None), ("tmax", None))):
        sel = np.arange(len(rays)) % 6 == k
        if axis is None:
            nan[field][sel] = np.nan
        else:
            nan[field][sel, axis] = np.nan
    nan_ref = E.trace(nan)
    assert (nan_ref["geom_id"] == INVALID).all()
    assert _check(E, nan, nan_ref, _seeds(ref["geom_id"], ref["prim_id"])) == 0
    E.close()


def test_raygen_seed_ties(emu):
    """a tied hint (same t, larger (geomID, primID)) is taken alike by both, and the traversal from it still returns the smaller IDs"""
    from test_gpu_parity import _tie_scene
    sb = _tie_scene()
    E = _emu(sb.desc())
    rays = scenes.primary_rays(64, 40.0, (0, 0, -3.0))
    ref = E.trace(rays)
    hit = ref["geom_id"] != INVALID
    assert hit.any() and (ref["geom_id"][hit] == 0).all()
    n = len(rays)
    for gg, pp in ((0, 1), (1, 0), (2, 0), (2, 1)):
        assert _check(E, rays, ref, _seeds(np.full(n, gg), np.full(n, pp))) > 0
    E.close()
