/* kz_refit.h -- accel refit: new boxes for the tree that kzgpu_accel_build made, after the vertices moved (kzgpu_mesh_update).
 *
 *   kz_refit_tri       re-gathers one 48-byte triangle record from the vertex records: the (geomID, primID) it carries in p0.w / p1.w
 *                      pick the index record, p0..p2 are read exactly as k_gather_tris reads them (same floats, same order)
 *   kz_refit_node      one wide node: the exact box of every used slot (a leaf slot: min/max of its <= 3 triangle records; an internal
 *                      slot: the box of node child_base + rank that the previous, deeper level computed), their union as the node box,
 *                      then k_collapse's quantisation (kz_lbvh.cuh) of every slot box in that frame
 *   kz_refit_levels    the level ranges of a node array emitted level by level (both builders do)
 *
 * Only origin, exponents and q-bytes of a node are rewritten; imask, trimask, child_base, tri_base, magic and the zeroed empty slots stay
 * as built.  Min / max are exact, so the result depends neither on the order in which nodes or levels' items run nor on the device.
 * A triangle that the builder referenced from two leaves with clipped boxes (pre-splitting) gets its whole box in both: looser, still
 * conservative.  Why the traversal still returns the hits of a fresh build: DESIGN.md section 3, "Refit".
 *
 * The KZ_HD functions are compiled by g++ for tests/hostemu (refit_emu.cpp) as well; kz_refit.cuh wraps them in kernels. */
#ifndef KZ_REFIT_H
#define KZ_REFIT_H
#include "kz_scene.h"
#include <vector>

struct KzBox { float lo[3], hi[3]; };

KZ_HD void kz_box_empty(KzBox &b) {
    for (int a = 0; a < 3; ++a) { b.lo[a] = kz_u2f(0x7f800000u); b.hi[a] = kz_u2f(0xff800000u); }
}
KZ_HD void kz_box_grow(KzBox &b, const KzBox &o) {
    for (int a = 0; a < 3; ++a) { b.lo[a] = fminf(b.lo[a], o.lo[a]); b.hi[a] = fmaxf(b.hi[a], o.hi[a]); }
}

/* Record `i` of `tris` from the current vertex records; returns its largest |coordinate|. */
KZ_HD float kz_refit_tri(const KzMeshRec *meshes, const KzVertex *vertices, const KzU4 *indices, KzF4 *tris, uint32_t i) {
    KzF4 *o = tris + 3 * (size_t)i;
    const uint32_t geom = kz_f2u(o[0].w), prim = kz_f2u(o[1].w);
    const KzMeshRec m = meshes[geom];
    const KzU4 t = indices[(size_t)m.index_offset + prim];
    const uint32_t vi[3] = {t.x, t.y, t.z};
    float mabs = 0.f;
    for (int k = 0; k < 3; ++k) {
        const KzVertex &v = vertices[(size_t)m.vertex_offset + vi[k]];
        KzF4 r; r.x = v.px; r.y = v.py; r.z = v.pz;
        r.w = k == 0 ? kz_u2f(geom) : (k == 1 ? kz_u2f(prim) : 0.f);
        o[k] = r;
        mabs = fmaxf(mabs, fmaxf(fabsf(r.x), fmaxf(fabsf(r.y), fabsf(r.z))));
    }
    return mabs;
}

/* Box of a refitted triangle record (any of its three vertices may be read in any order: min / max are exact). */
KZ_HD KzBox kz_record_box(const KzF4 *tris, uint32_t t) {
    const KzF4 *p = tris + 3 * (size_t)t;
    KzBox b;
    b.lo[0] = fminf(p[0].x, fminf(p[1].x, p[2].x)); b.hi[0] = fmaxf(p[0].x, fmaxf(p[1].x, p[2].x));
    b.lo[1] = fminf(p[0].y, fminf(p[1].y, p[2].y)); b.hi[1] = fmaxf(p[0].y, fmaxf(p[1].y, p[2].y));
    b.lo[2] = fminf(p[0].z, fminf(p[1].z, p[2].z)); b.hi[2] = fmaxf(p[0].z, fmaxf(p[1].z, p[2].z));
    return b;
}

/* Refits node `n` in place from the refitted triangle records and the boxes of its internal children (`boxes`, indexed by node);
 * returns the node's box (to be stored in boxes[n] for its parent). */
KZ_HD KzBox kz_refit_node(KzNode8 &n, const KzF4 *tris, const KzBox *boxes) {
    KzBox bx[8];
    KzBox nb; kz_box_empty(nb);
    uint32_t used = 0u;
    for (int s = 0; s < 8; ++s) {
        const uint32_t bits = (n.trimask >> (3 * s)) & 7u;
        if ((n.imask >> s) & 1u) {
            bx[s] = boxes[n.child_base + kz_popc((uint32_t)n.imask & ((1u << s) - 1u))];
        } else if (bits) {
            kz_box_empty(bx[s]);
            for (int k = 0; k < 3; ++k)
                if ((bits >> k) & 1u) kz_box_grow(bx[s], kz_record_box(tris, n.tri_base + kz_popc(n.trimask & ((1u << (3 * s + k)) - 1u))));
        } else continue;
        used |= 1u << s;
        kz_box_grow(nb, bx[s]);
    }
    if (!used) return nb;
    /* +0.f turns a -0 origin into +0: which zero fminf keeps is not specified, and the node bytes must not depend on it */
    n.px = nb.lo[0] + 0.f; n.py = nb.lo[1] + 0.f; n.pz = nb.lo[2] + 0.f;
    /* k_collapse's frame: smallest power of two 2^(e-127) with ceil(ext / 2^(e-127)) <= 255, e in [1, 254] */
    int e[3];
    for (int a = 0; a < 3; ++a) {
        const double ext = (double)nb.hi[a] - (double)nb.lo[a];
        int ee = 1 - 127;
        if (ext > 0.0) frexp(ext / 255.0, &ee);
        int biased = ee + 127;
        biased = biased < 1 ? 1 : (biased > 254 ? 254 : biased);
        while (biased < 254 && ceil(ext / ldexp(1.0, biased - 127)) > 255.0) ++biased;
        e[a] = biased;
    }
    n.ex = (uint8_t)e[0]; n.ey = (uint8_t)e[1]; n.ez = (uint8_t)e[2];
    uint8_t *qlo[3] = {n.qlox, n.qloy, n.qloz}, *qhi[3] = {n.qhix, n.qhiy, n.qhiz};
    for (int s = 0; s < 8; ++s) {
        if (!((used >> s) & 1u)) continue;
        for (int a = 0; a < 3; ++a) {
            const double sc = ldexp(1.0, e[a] - 127);
            const double lo = floor(((double)bx[s].lo[a] - (double)nb.lo[a]) / sc);
            const double hi = ceil(((double)bx[s].hi[a] - (double)nb.lo[a]) / sc);
            qlo[a][s] = (uint8_t)fmin(255.0, fmax(0.0, lo));
            qhi[a][s] = (uint8_t)fmin(255.0, fmax(0.0, hi));
        }
    }
    return nb;
}

/* Level l of a node array emitted level by level is [first[l], first[l + 1]): level 0 is the root, level l + 1 holds the internal
 * children of level l.  Derived from the masks of a host-resident array (the host SAH builder); false if the array is not laid out so. */
inline bool kz_refit_levels(const KzNode8 *nodes, uint32_t n_nodes, std::vector<uint32_t> &first) {
    first.assign(1, 0u);
    if (n_nodes == 0) return true;
    uint32_t lo = 0, hi = 1;
    while (lo < hi) {
        first.push_back(hi);
        uint64_t next = hi;
        for (uint32_t i = lo; i < hi; ++i) {
            const uint32_t k = kz_popc(nodes[i].imask);
            if (!k) continue;
            if ((uint64_t)nodes[i].child_base != next) return false;
            next += k;
        }
        if (next > n_nodes) return false;
        lo = hi; hi = (uint32_t)next;
    }
    return first.back() == n_nodes;
}

#endif
