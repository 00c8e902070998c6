/* tests/hostemu/seed_emu.cpp -- DEVELOPMENT/TEST HARNESS, NOT A PRODUCT PATH.
 *
 * emu.cpp (the device routines compiled for the host) plus the traversal seeded with a closest-hit hint (kz_trav_seed,
 * kz_traverse.h), as k_extend<true> seeds every primary ray with the triangle its pixel hit last.  Built as its own library
 * (seed_emu.py) so that the CPU suite can check that a seeded traversal returns the same hits as an unseeded one.
 */
#include "emu.cpp"

extern "C" {

/* kz_trace with a hint per ray: seeds = n (geomID, primID) pairs, KZ_INVALID_ID for none; *seeded = the number of hints the ray hit. */
int kzemu_trace_seeded(kzemu *e, const kz_ray *rays, const uint32_t *seeds, size_t n, kz_hit *hits, uint64_t *seeded) {
    const KzScene &sc = e->hs.sc;
    std::atomic<uint64_t> a_seeded{0};
    pfor(n, [&](size_t b, size_t en) {
        KzStackRef stk;
        uint64_t k = 0;
        for (size_t i = b; i < en; ++i) {
            const kz_ray &r = rays[i];
            KzTrav t;
            kz_trav_init(sc, t, r.o[0], r.o[1], r.o[2], r.d[0], r.d[1], r.d[2], r.tmin, r.tmax);
            k += kz_trav_seed(sc, t, seeds[2 * i], seeds[2 * i + 1]) ? 1u : 0u;
            const KzHit h = kz_trace(sc, stk, r.o[0], r.o[1], r.o[2], r.d[0], r.d[1], r.d[2], r.tmin, r.tmax, false, seeds[2 * i], seeds[2 * i + 1]);
            hits[i].t = h.t; hits[i].u = h.u; hits[i].v = h.v; hits[i].prim_id = h.prim; hits[i].geom_id = h.geom;
        }
        a_seeded += k;
    });
    if (seeded) *seeded = a_seeded.load();
    return KZ_OK;
}

/* Node steps and triangle tests of the plain per-ray loop (as kzemu_trace_stats), each ray seeded as above: out = {node steps, triangle tests}. */
int kzemu_trace_stats_seeded(kzemu *e, const kz_ray *rays, const uint32_t *seeds, size_t n, uint64_t *out) {
    const KzScene &sc = e->hs.sc;
    std::atomic<uint64_t> a_nodes{0}, a_tris{0};
    pfor(n, [&](size_t b, size_t en) {
        KzStackRef stk;
        uint64_t nodes = 0, tris = 0;
        for (size_t i = b; i < en; ++i) {
            const kz_ray &r = rays[i];
            KzTrav t; KzLocalStack ls;
            kz_trav_init(sc, t, r.o[0], r.o[1], r.o[2], r.d[0], r.d[1], r.d[2], r.tmin, r.tmax);
            if (sc.n_nodes == 0) continue;
            kz_trav_seed(sc, t, seeds[2 * i], seeds[2 * i + 1]);
            for (;;) {
                if (t.ng_y > 0x00FFFFFFu) { kz_trav_node(sc, t, stk, ls); ++nodes; }
                while (t.tg_y != 0u) { kz_trav_tri(sc, t); ++tris; }
                if (t.ng_y <= 0x00FFFFFFu) { if (t.sp == 0) break; kz_trav_pop(t, stk, ls); }
            }
        }
        a_nodes += nodes; a_tris += tris;
    });
    out[0] = a_nodes; out[1] = a_tris;
    return KZ_OK;
}

}  // extern "C"
