/* tests/hostemu/raygen_seed_emu.cpp -- DEVELOPMENT/TEST HARNESS, NOT A PRODUCT PATH.
 *
 * emu.cpp (the device routines compiled for the host) plus the two halves of the primary-hit seed as the device runs them: k_raygen
 * tests the hint on the ray it generated (kz_seed_hit) and k_extend<true> installs the result in a fresh traversal (kz_trav_preset).
 * Built as its own library (raygen_seed_emu.py) so that the CPU suite can hold that split to kz_trav_seed, bit for bit.
 */
#include "emu.cpp"

extern "C" {

/* Per ray and hint (seeds = n (geomID, primID) pairs): pure[i] = kz_seed_hit on the ray's own (o, d, tmin, tmax), trav[i] = the best hit
 * kz_trav_seed leaves in a fresh traversal of the ray (t = tmax and invalid IDs if it took no seed); taken[i] = bit 0: kz_seed_hit hit,
 * bit 1: kz_trav_seed seeded, bit 2: kz_trav_preset installed pure[i] in a fresh traversal. */
int kzemu_seed_split(kzemu *e, const kz_ray *rays, const uint32_t *seeds, size_t n, kz_hit *pure, kz_hit *trav, uint8_t *taken) {
    const KzScene &sc = e->hs.sc;
    pfor(n, [&](size_t b, size_t en) {
        for (size_t i = b; i < en; ++i) {
            const kz_ray &r = rays[i];
            KzHit h; h.t = h.u = h.v = 0.f; h.prim = h.geom = KZ_INVALID_ID;          /* as k_raygen starts it */
            const bool hit = kz_seed_hit(sc, r.o[0], r.o[1], r.o[2], r.d[0], r.d[1], r.d[2], r.tmin, r.tmax, seeds[2 * i], seeds[2 * i + 1], h);
            KzTrav t;
            kz_trav_init(sc, t, r.o[0], r.o[1], r.o[2], r.d[0], r.d[1], r.d[2], r.tmin, r.tmax);
            const bool seeded = kz_trav_seed(sc, t, seeds[2 * i], seeds[2 * i + 1]);
            KzTrav p;
            kz_trav_init(sc, p, r.o[0], r.o[1], r.o[2], r.d[0], r.d[1], r.d[2], r.tmin, r.tmax);
            const bool installed = kz_trav_preset(p, h);
            pure[i].t = h.t; pure[i].u = h.u; pure[i].v = h.v; pure[i].prim_id = h.prim; pure[i].geom_id = h.geom;
            trav[i].t = t.best.t; trav[i].u = t.best.u; trav[i].v = t.best.v; trav[i].prim_id = t.best.prim; trav[i].geom_id = t.best.geom;
            taken[i] = (uint8_t)((hit ? 1u : 0u) | (seeded ? 2u : 0u) | (installed ? 4u : 0u));
        }
    });
    return KZ_OK;
}

/* The closest hit of the plain per-ray loop started from a preset (presets = n kz_hit records, as k_raygen leaves them; geom_id
 * KZ_INVALID_ID: none), installed with kz_trav_preset as k_extend<true> does. */
int kzemu_trace_preset(kzemu *e, const kz_ray *rays, const kz_hit *presets, size_t n, kz_hit *hits) {
    const KzScene &sc = e->hs.sc;
    pfor(n, [&](size_t b, size_t en) {
        KzStackRef stk;
        for (size_t i = b; i < en; ++i) {
            const kz_ray &r = rays[i];
            KzTrav t; KzLocalStack ls;
            kz_trav_init(sc, t, r.o[0], r.o[1], r.o[2], r.d[0], r.d[1], r.d[2], r.tmin, r.tmax);
            KzHit h; h.t = presets[i].t; h.u = presets[i].u; h.v = presets[i].v; h.prim = presets[i].prim_id; h.geom = presets[i].geom_id;
            kz_trav_preset(t, h);
            if (t.ng_y != 0u) for (;;) {
                if (t.ng_y > 0x00FFFFFFu) kz_trav_node(sc, t, stk, ls);
                while (t.tg_y != 0u) kz_trav_tri(sc, t);
                if (t.ng_y <= 0x00FFFFFFu) { if (t.sp == 0) break; kz_trav_pop(t, stk, ls); }
            }
            hits[i].t = t.best.t; hits[i].u = t.best.u; hits[i].v = t.best.v; hits[i].prim_id = t.best.prim; hits[i].geom_id = t.best.geom;
        }
    });
    return KZ_OK;
}

}  // extern "C"
