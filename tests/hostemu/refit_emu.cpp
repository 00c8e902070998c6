/* tests/hostemu/refit_emu.cpp -- DEVELOPMENT/TEST HARNESS, NOT A PRODUCT PATH.
 *
 * emu.cpp (the device routines compiled for the host) plus the accel refit of kz_refit.h, run on the emulation's host-SAH accel the
 * way kzgpu_accel_refit runs it on the device: every triangle record re-gathered, then the levels deepest first.  Built as its own
 * library (refit_emu.py) so that the CPU suite can check a refitted accel against the oracle on the moved scene.
 */
#include "emu.cpp"
#include "../../nano-kazen_b200/csrc/kz_refit.h"
#include <memory>

extern "C" {

/* Replaces the emulation's scene by `d` (same meshes, vertex and triangle counts, new positions) and refits the accel it built for
 * the old one.  KZ_ERR_INVALID if `d` is not the same topology, KZ_ERR_STATE if the accel is not laid out level by level. */
int kzemu_refit(kzemu *e, const kz_scene_desc *d) {
    std::unique_ptr<KzHostScene> hs(new KzHostScene());
    if (!hs->flatten(d)) { fprintf(stderr, "kzemu: %s\n", hs->error.c_str()); return KZ_ERR_INVALID; }
    if (hs->meshes.size() != e->hs.meshes.size() || hs->total_vertices != e->hs.total_vertices || hs->total_triangles != e->hs.total_triangles) return KZ_ERR_INVALID;
    for (size_t g = 0; g < hs->meshes.size(); ++g)
        if (hs->meshes[g].vertex_offset != e->hs.meshes[g].vertex_offset) return KZ_ERR_INVALID;
    std::vector<uint32_t> L;
    if (!kz_refit_levels(e->bvh.nodes.data(), (uint32_t)e->bvh.nodes.size(), L)) return KZ_ERR_STATE;
    e->hs.meshes.swap(hs->meshes); e->hs.vertices.swap(hs->vertices); e->hs.indices.swap(hs->indices); e->hs.light_cdf.swap(hs->light_cdf);
    e->hs.light_bounds.swap(hs->light_bounds); e->hs.tris.swap(hs->tris);
    for (int a = 0; a < 3; ++a) { e->hs.sc.inv_light_lo[a] = hs->sc.inv_light_lo[a]; e->hs.sc.inv_light_hi[a] = hs->sc.inv_light_hi[a]; }
    e->hs.finalize();
    const KzScene &sc = e->hs.sc;
    float mabs = 0.f;
    for (uint32_t i = 0; i < (uint32_t)(e->bvh.tris.size() / 3); ++i) mabs = fmaxf(mabs, kz_refit_tri(sc.meshes, sc.vertices, sc.indices, e->bvh.tris.data(), i));
    std::vector<KzBox> boxes(e->bvh.nodes.size());
    for (int l = (int)L.size() - 2; l >= 0; --l)
        for (uint32_t i = L[(size_t)l]; i < L[(size_t)l + 1]; ++i) boxes[i] = kz_refit_node(e->bvh.nodes[i], e->bvh.tris.data(), boxes.data());
    e->hs.sc.nodes = e->bvh.nodes.data(); e->hs.sc.tris = e->bvh.tris.data();
    e->hs.sc.scene_max_abs = mabs;
    return KZ_OK;
}

/* The emulation's accel: n_nodes 80-byte nodes and 3 * n_tris float4 (sizes from kzemu_bvh_info). */
int kzemu_accel_dump(kzemu *e, void *nodes, void *tris) {
    memcpy(nodes, e->bvh.nodes.data(), e->bvh.nodes.size() * sizeof(KzNode8));
    memcpy(tris, e->bvh.tris.data(), e->bvh.tris.size() * sizeof(KzF4));
    return KZ_OK;
}

/* max |coordinate| the traversal slack is scaled with */
int kzemu_scene_max_abs(kzemu *e, float *out) { *out = e->hs.sc.scene_max_abs; return KZ_OK; }

}  // extern "C"
