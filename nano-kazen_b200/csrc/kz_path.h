/* kz_path.h -- the wavefront stages of PathMisIntegrator::Li as per-item routines over SoA
 * path state.  One "item" = one path slot.  Stage order per bounce b = 0..maxDepth:
 *
 *   raygen  (b = 0 only)  renderer.cpp:20-33 + camera.cpp:70-91,191-223
 *   extend                Scene::rayIntersect (closest hit) [+ the one-shot invisible-light
 *                         re-trace of integrator.cpp:214-219 when b == 0]
 *   shade                 integrator.cpp:224-334 for one loop iteration: light hit / miss /
 *                         RR / NEE set-up / regularisation / BSDF sampling
 *   shadow                integrator.cpp:259-294: closest-hit walk through invisible lights,
 *                         then Li += pending
 *   accumulate (end)      ImageBlock::put, block.cpp:56-85
 *
 * The reference's loop is   [hit] -> { light? RR NEE BSDF-sample trace -> miss? light-MIS depth++ }.
 * Here iteration k's tail (miss / light-MIS weight / depth++) runs at the head of shade(b = k+1),
 * so there are maxDepth+1 extend passes and the last shade only resolves the final ray.
 */
#ifndef KZ_PATH_H
#define KZ_PATH_H
#include "kz_env.h"
#include "kz_texlod.h"

/* Path state: three 64-byte blocks per slot, grouped by which stage touches what, so that every access of a stage is a
 * whole 32-byte DRAM sector (slots are visited in queue order, i.e. scattered: the former one-array-per-field layout moved a
 * 32-byte sector for every 16- or 4-byte field, 12 sectors per shaded vertex instead of 5).  All members are 16-byte aligned,
 * so a record moves as 128-bit loads / stores.
 *   A = ray (read by extend, written by shade)      | hit (written by extend, read by shade)
 *   B = throughput|eta, Li|bsdfPdf of the last sampled direction (shade, shadow, accumulate) | sampler state, accumulatedRoughness
 *   C = shadow ray d|tmax, pending rgb|tmin (origin = A.ray.o); 32 bytes
 * Not stored: bsdfWeight (only lives between the tail of one loop iteration and the head of the next, both inside one shade
 * pass) and the pixel sample position (recomputed from the addressable sampler when the path is splatted). */
struct alignas(16) KzRayRec { KzF4 o, d; };                          /* o.xyz tmin | d.xyz tmax */
/* Hit record.  Between k_raygen and k_extend<true>, with primary-hit hints on, it holds the seed of the primary ray (kz_seed_hit; an
 * invalid hit if there is none) and `pix` carries the film pixel the hint goes back to (as KzSmpRec::pix; 0xFFFFFFFF on padding lanes).
 * No other stage reads `pix`: it is 0 in every hit that extend stores. */
struct alignas(16) KzHitRec { float t, u, v; uint32_t prim, geom, pix, pad1, pad2; };
struct alignas(64) KzBlockA { KzRayRec ray; KzHitRec hit; };
struct alignas(16) KzRadRec { KzF4 thr, L; };                        /* throughput rgb, eta | Li rgb, bsdfPdf (< 0: discrete) */
struct alignas(16) KzSmpRec { uint64_t rng_state, rng_inc; uint32_t dim, pix /* px | py << 16 */, sidx; float acc_rough; };
struct alignas(64) KzBlockB { KzRadRec rad; KzSmpRec smp; };
struct alignas(16) KzShdRec { KzF4 d, pending; };                    /* d.xyz tmax | NEE rgb awaiting visibility, tmin */
struct alignas(32) KzBlockC { KzShdRec shd; };
static_assert(sizeof(KzBlockA) == 64 && sizeof(KzBlockB) == 64 && sizeof(KzBlockC) == 32, "path state blocks are whole sectors");

struct KzPathState {
    KzBlockA *a;
    KzBlockB *b;
    KzBlockC *c;
};
KZ_HD KzHitRec mk_hit_rec(const KzHit &h) { KzHitRec r; r.t = h.t; r.u = h.u; r.v = h.v; r.prim = h.prim; r.geom = h.geom; r.pix = r.pad1 = r.pad2 = 0u; return r; }

struct KzCounters {
    unsigned long long paths, rays_ext, rays_shadow, vertices, rays_seeded;     /* rays_seeded: primary rays that started from a hit hint */
};

#define KZ_SHADE_CONTINUE 1u   /* extension ray written, path goes to the next extend pass */
#define KZ_SHADE_SHADOW 2u     /* shadow ray + pending contribution written               */

/* `bsdf->sample(bRec, sampler->next1D(), sampler->next2D())` (integrator.cpp:122,168,307): GCC evaluates the two draws right to left
 * (next2D first), see oracle/kzo.cpp; KZ_ARG_ORDER_LTR=1 restores the textual order. */
#ifndef KZ_ARG_ORDER_LTR
#define KZ_ARG_ORDER_LTR 0
#endif
#if KZ_ARG_ORDER_LTR
#define KZ_DRAW_BSDF_SAMPLES(sc, sm, s1, s2) const float s1 = kz_next1d(sc, sm); const kz2 s2 = kz_next2d(sc, sm)
#else
#define KZ_DRAW_BSDF_SAMPLES(sc, sm, s1, s2) const kz2 s2 = kz_next2d(sc, sm); const float s1 = kz_next1d(sc, sm)
#endif

KZ_HD float power_heuristic(float a, float b) { a *= a; b *= b; return a > 0.f ? a / (a + b) : 0.f; }

KZ_HD kz3 xform_point(const float *M, kz3 p) {
    float r0 = M[0] * p.x + M[1] * p.y + M[2] * p.z + M[3];
    float r1 = M[4] * p.x + M[5] * p.y + M[6] * p.z + M[7];
    float r2 = M[8] * p.x + M[9] * p.y + M[10] * p.z + M[11];
    float r3 = M[12] * p.x + M[13] * p.y + M[14] * p.z + M[15];
    return mk3(r0 / r3, r1 / r3, r2 / r3);
}
KZ_HD kz3 xform_vector(const float *M, kz3 v) {
    return mk3(M[0] * v.x + (M[1] * v.y + M[2] * v.z), M[4] * v.x + (M[5] * v.y + M[6] * v.z), M[8] * v.x + (M[9] * v.y + M[10] * v.z));
}

/* camera.cpp:70-91 / 191-223 */
KZ_HD void kz_camera_ray(const kz_camera_desc &c, kz2 samplePosition, kz2 apertureSample, KzF4 &ro, KzF4 &rd) {
    const float invW = 1.0f / (float)c.width, invH = 1.0f / (float)c.height;
    kz3 nearP = xform_point(c.sample_to_camera, mk3(samplePosition.x * invW, samplePosition.y * invH, 0.0f));
    kz3 o, d;
    if (c.type == KZ_CAM_THINLENS) {
        kz2 tmp = square_to_uniform_disk(apertureSample);
        kz3 apertureP = mk3(tmp.x * c.aperture_radius, tmp.y * c.aperture_radius, 0.0f);
        kz3 focusP = nearP * (c.focus_distance / nearP.z);
        d = normalized(focusP - apertureP);
        o = xform_point(c.camera_to_world, apertureP);
    } else {
        d = normalized(nearP);
        o = xform_point(c.camera_to_world, mk3(0.f, 0.f, 0.f));
    }
    const float invZ = 1.0f / d.z;
    kz3 dw = xform_vector(c.camera_to_world, d);
    ro.x = o.x; ro.y = o.y; ro.z = o.z; ro.w = c.near_clip * invZ;
    rd.x = dw.x; rd.y = dw.y; rd.z = dw.z; rd.w = c.far_clip * invZ;
}

KZ_HD KzF4 mkf4(float x, float y, float z, float w) { KzF4 r; r.x = x; r.y = y; r.z = z; r.w = w; return r; }

KZ_HD KzSmpRec kz_sampler_save(const KzSampler &sm, float acc_rough) {
    KzSmpRec r; r.rng_state = sm.state; r.rng_inc = sm.inc; r.dim = sm.dim;
    r.pix = (uint32_t)sm.px | ((uint32_t)sm.py << 16); r.sidx = sm.sample_index; r.acc_rough = acc_rough;
    return r;
}
KZ_HD void kz_sampler_load(KzSampler &sm, const KzSmpRec &r) {
    sm.state = r.rng_state; sm.inc = r.rng_inc; sm.dim = r.dim;
    sm.px = (int32_t)(r.pix & 0xFFFFu); sm.py = (int32_t)(r.pix >> 16); sm.sample_index = r.sidx;
}

/* ---- raygen -------------------------------------------------------------------------------- */
/* Writes the path's camera ray and its throughput / sampler state; returns the ray. */
KZ_HD KzRayRec kz_raygen_item(const KzScene &sc, const KzPathState &st, uint32_t slot, int px, int py, uint32_t sample_index) {
    KzSampler sm;
    kz_sampler_start(sc, sm, px, py, sample_index);
    kz2 pix = kz_next_pixel2d(sc, sm);
    kz2 pixelSample = mk2((float)px + pix.x, (float)py + pix.y);
    kz2 aperture = kz_next2d(sc, sm);
    KzF4 ro, rd;
    kz_camera_ray(sc.camera, pixelSample, aperture, ro, rd);
    KzRayRec ray; ray.o = ro; ray.d = rd;
    st.a[slot].ray = ray;
    KzBlockB B; B.rad.thr = mkf4(1.f, 1.f, 1.f, 1.f); B.rad.L = mkf4(0.f, 0.f, 0.f, 0.f); B.smp = kz_sampler_save(sm, 0.f);
    st.b[slot] = B;
    return ray;
}

KZ_HD int kz_classify(const KzScene &sc, uint32_t geom) {
    if (sc.integrator.type != KZ_INTEGRATOR_PATH_MIS) return KZ_CLASS_GENERIC;     /* the other integrators are not material sorted */
    if (geom == KZ_INVALID_ID) return KZ_CLASS_TERMINAL;
    const KzMeshRec m = sc.meshes[geom];
    if (m.flags & KZ_MESH_IS_LIGHT) return KZ_CLASS_TERMINAL;
    const int t = sc.bsdfs[m.bsdf].type;
    return t == KZ_BSDF_DIFFUSE ? KZ_CLASS_DIFFUSE : (t == KZ_BSDF_KISS ? KZ_CLASS_KISS : (t == KZ_BSDF_NORMALMAP ? KZ_CLASS_NORMALMAP : KZ_CLASS_GENERIC));
}

/* ---- extend -------------------------------------------------------------------------------- */
/* Traces the path's current ray, stores the hit, returns the material class of the hit. */
KZ_HD int kz_extend_item(const KzScene &sc, const KzStackRef &stk, const KzPathState &st, uint32_t slot, int bounce, KzCounters &cnt) {
    const KzRayRec ray = st.a[slot].ray;
    const KzF4 ro = ray.o, rd = ray.d;
    KzHit h = kz_trace(sc, stk, ro.x, ro.y, ro.z, rd.x, rd.y, rd.z, ro.w, rd.w, false);
    cnt.rays_ext += 1;
    if (bounce == 0 && h.geom != KZ_INVALID_ID && sc.integrator.type == KZ_INTEGRATOR_PATH_MIS) {
        const KzMeshRec m = sc.meshes[h.geom];
        if ((m.flags & KZ_MESH_IS_LIGHT) && !(m.flags & KZ_MESH_LIGHT_VISIBLE)) {
            /* integrator.cpp:214-219: one re-trace from its.p + eps*d; a miss keeps the light hit */
            KzIts its; its.acc_rough = 0.f;
            fill_intersection(sc, h, its, mk3(0.f));
            const float eps = sc.integrator.trace_bias;
            const kz3 d = mk3(rd.x, rd.y, rd.z);
            const kz3 o = its.p + eps * d;
            KzHit h2 = kz_trace(sc, stk, o.x, o.y, o.z, d.x, d.y, d.z, KZ_EPSILON, KZ_INF, false);
            cnt.rays_ext += 1;
            if (h2.geom != KZ_INVALID_ID) h = h2;
        }
    }
    st.a[slot].hit = mk_hit_rec(h);
    return kz_classify(sc, h.geom);
}

/* ---- emitter sampling: Scene::getRandomLight (scene.h:45-56) + Mesh::sample (mesh.cpp:108-133) + AreaLight::sample / pdf
 *      (light.cpp:21-51).  u_pick, u_tri, u_b1, u_b2: the four 1-D draws in the order Li makes them. ------------------------ */
struct KzEmitterSample {
    int32_t mesh;        /* scene mesh index of the picked emitter */
    int32_t light;       /* its kz_light_desc */
    kz3 p, n, wi;        /* sampled point, its (unnormalised) normal, direction ref -> p */
    float dist, pdf;     /* |p - ref|, solid-angle density (0: not usable); the pick probability 1/n_lights is NOT included */
};
/* `index`: the picked emitter, into light_meshes */
KZ_HD KzEmitterSample kz_sample_emitter_at(const KzScene &sc, uint32_t index, kz3 ref, float u_tri, float u_b1, float u_b2) {
    KzEmitterSample es;
    es.mesh = sc.light_meshes[index];
    const KzMeshRec lm = sc.meshes[es.mesh];
    es.light = lm.light;
    /* Mesh::sample, mesh.cpp:108-133 */
    const uint32_t tri = cdf_sample(sc.light_cdf + lm.cdf_offset, lm.n_triangles, u_tri);
    const float su0 = sqrtf(u_b1);
    const float u = 1 - su0;
    const float v = u_b2 * su0;
    const KzU4 F = sc.indices[(size_t)lm.index_offset + tri];
    const KzVertex lv0 = kz_vertex(sc, lm, F.x), lv1 = kz_vertex(sc, lm, F.y), lv2 = kz_vertex(sc, lm, F.z);
    const kz3 p0 = kz_vpos(lv0), p1 = kz_vpos(lv1), p2 = kz_vpos(lv2);
    es.p = p0 + u * (p1 - p0) + v * (p2 - p0);
    if (lm.flags & KZ_MESH_HAS_NORMALS) {
        const kz3 n0 = kz_vnrm(lv0), n1 = kz_vnrm(lv1), n2 = kz_vnrm(lv2);
        es.n = n0 + u * (n1 - n0) + v * (n2 - n0);          /* not normalised, mesh.cpp:128-129 */
    } else {
        es.n = normalized(cross(p1 - p0, p2 - p0));
    }
    /* AreaLight::sample, light.cpp:21-34 */
    es.wi = normalized(es.p - ref);
    es.dist = norm(es.p - ref);
    es.pdf = light_pdf(lm.inv_area, ref, es.p, es.n, es.wi);
    return es;
}
KZ_HD KzEmitterSample kz_sample_emitter(const KzScene &sc, kz3 ref, float u_pick, float u_tri, float u_b1, float u_b2) {
    const uint32_t nl = (uint32_t)sc.n_light_meshes;
    uint32_t index = (uint32_t)floorf((float)nl * u_pick);
    if (index > nl - 1) index = nl - 1;
    return kz_sample_emitter_at(sc, index, ref, u_tri, u_b1, u_b2);
}

/* ---- shade --------------------------------------------------------------------------------- */
KZ_HD_NOINLINE uint32_t kz_shade_alt_item(const KzScene &sc, const KzPathState &st, uint32_t slot, int bounce, KzCounters &cnt);

/* CLS = material class of the queue this item was sorted into (-1: unknown, resolve at run time).
 * ENV = the environment is a light with table `env` (kz_env.h): next-event estimation picks it as light n_light_meshes with
 * probability 1 / (n_light_meshes + 1), and a BSDF-sampled ray that escapes is weighted against its density.  ENV = false is the
 * reference estimator and does not read `env`.
 * FILT = uv-mode image lookups of the vertex's textures are filtered by its footprint (kz_texlod.h), estimated from the camera constants
 * `lod`; FILT = false reads level 0 as the reference does and does not read `lod`. */
template <int CLS = -1, bool ENV = false, bool FILT = false>
KZ_HD uint32_t kz_shade_item(const KzScene &sc, const KzPathState &st, uint32_t slot, int bounce, KzCounters &cnt, const KzEnvTable &env = KzEnvTable{},
                             const KzTexLod &lod = KzTexLod{}) {
    if ((CLS < 0 || CLS == KZ_CLASS_GENERIC) && sc.integrator.type != KZ_INTEGRATOR_PATH_MIS) return kz_shade_alt_item(sc, st, slot, bounce, cnt);
    const KzBlockA A = st.a[slot];
    const KzF4 ro = A.ray.o, rd = A.ray.d;
    const kz3 rayO = mk3(ro.x, ro.y, ro.z), rayD = mk3(rd.x, rd.y, rd.z);
    KzHit h; h.t = A.hit.t; h.u = A.hit.u; h.v = A.hit.v; h.prim = A.hit.prim; h.geom = A.hit.geom;
    const KzRadRec rad = st.b[slot].rad;
    const KzF4 thr4 = rad.thr, L4 = rad.L;
    kz3 throughput = mk3(thr4.x, thr4.y, thr4.z), L = mk3(L4.x, L4.y, L4.z);
    float eta = thr4.w, bsdfWeight = 1.f;       /* integrator.cpp:207: only changes when a sampled ray lands on a light (below) */
    const float prevBsdfPdf = L4.w;
    const KzIntegrator I = sc.integrator;

    if (CLS <= KZ_CLASS_TERMINAL && h.geom == KZ_INVALID_ID) {     /* material-class queues never hold misses */
        /* bounce 0: camera rays never see the background (integrator.cpp:210-212);
         * later: Li += throughput * background(ray.d) (integrator.cpp:315-318) */
        if (bounce > 0) {
            if (ENV) L += throughput * kz_background(sc, rayD) * (prevBsdfPdf < 0.f ? 1.f : power_heuristic(prevBsdfPdf, kz_env_pdf(env, rayD)));
            else L += throughput * kz_background(sc, rayD);
            st.b[slot].rad.L = mkf4(L.x, L.y, L.z, bsdfWeight);
        }
        return 0u;
    }
    KzIts its; its.acc_rough = 0.f;
    fill_intersection(sc, h, its, mk3(0.f));
    const KzMeshRec mesh = sc.meshes[its.mesh];
    const bool isLight = (mesh.flags & KZ_MESH_IS_LIGHT) != 0;
    if (bounce > 0 && isLight) {   /* integrator.cpp:322-327 */
        const kz3 wi = normalized(its.p - rayO);
        const float lightPdf_ = light_pdf(mesh.inv_area, rayO, its.p, its.sh.n, wi);
        bsdfWeight = prevBsdfPdf < 0.f ? 1.f : power_heuristic(prevBsdfPdf, lightPdf_);
    }
    if (bounce >= I.max_depth) return 0u;          /* depth++ ; while (depth < maxDepth) */
    if (isLight) {       /* integrator.cpp:226-231 */
        const kz3 wi = normalized(its.p - rayO);
        const float cosTheta = dot(its.sh.n, -wi);
        if (cosTheta > 0.f) {
            const kz_light_desc l = sc.lights[mesh.light];
            L += bsdfWeight * throughput * mk3(l.radiance[0], l.radiance[1], l.radiance[2]);
            st.b[slot].rad.L = mkf4(L.x, L.y, L.z, bsdfWeight);
        }
        return 0u;
    }
    if (CLS == KZ_CLASS_TERMINAL) return 0u;      /* that queue only holds misses and light hits */

    KzSampler sm;
    {
        const KzSmpRec smp = st.b[slot].smp;
        kz_sampler_load(sm, smp);
        its.acc_rough = smp.acc_rough;
    }

    if (bounce >= 3) {   /* integrator.cpp:237-244 */
        const float probability = fminf(maxcoeff(throughput) * eta * eta, 0.95f);
        if (probability <= kz_next1d(sc, sm)) return 0u;
        throughput = throughput / probability;
    }
    cnt.vertices += 1;
    uint32_t flags = 0u;
    KzUvDiff duv{0.f, 0.f, 0.f, 0.f};
    if (FILT) duv = kz_its_footprint(sc, lod, h, its);
    const KzBsdfCtx<FILT> bc = bsdf_ctx<CLS, FILT>(sc, its, duv);
    const kz3 wiLocal = to_local(its.sh, -rayD);
    const float eps = I.trace_bias;

    /* ---- light sampling, integrator.cpp:247-294 ---- */
    const float rnd = kz_next1d(sc, sm);
    if (ENV) {
        /* the reference's draws, whichever light is picked; the environment uses the second and third and leaves the fourth */
        const uint32_t nl = (uint32_t)sc.n_light_meshes + 1u;
        const float u_tri = kz_next1d(sc, sm);
        const float u_b1 = kz_next1d(sc, sm);
        const float u_b2 = kz_next1d(sc, sm);
        uint32_t index = (uint32_t)floorf((float)nl * rnd);
        if (index > nl - 1) index = nl - 1;
        if (index == nl - 1) {
            const kz3 lwi = kz_env_sample(env, u_tri, u_b1);
            const float lpdf = kz_env_pdf(env, lwi);
            if (lpdf > 0.f && !isnan(lpdf) && !isinf(lpdf)) {
                const kz3 Ls = kz_background(sc, lwi) / lpdf * (float)nl;
                kz3 f; float bsdfPdf;
                bsdf_eval_pdf(bc, its, wiLocal, to_local(its.sh, lwi), &f, &bsdfPdf);
                const kz3 contrib = throughput * Ls * f * power_heuristic(lpdf, bsdfPdf);
                if (!iszero(contrib)) {
                    KzShdRec shd; shd.d = mkf4(lwi.x, lwi.y, lwi.z, KZ_INF); shd.pending = mkf4(contrib.x, contrib.y, contrib.z, eps);
                    st.c[slot].shd = shd;
                    flags |= KZ_SHADE_SHADOW;
                }
            }
        } else {
            const KzEmitterSample es = kz_sample_emitter_at(sc, index, its.p, u_tri, u_b1, u_b2);
            if (es.pdf > 0.f && !isnan(es.pdf) && !isinf(es.pdf)) {
                const kz_light_desc l = sc.lights[es.light];
                const kz3 Ls = mk3(l.radiance[0], l.radiance[1], l.radiance[2]) / es.pdf / (1.f / (float)nl);
                kz3 f; float bsdfPdf;
                bsdf_eval_pdf(bc, its, wiLocal, to_local(its.sh, es.wi), &f, &bsdfPdf);
                const kz3 contrib = throughput * Ls * f * power_heuristic(es.pdf, bsdfPdf);
                if (!iszero(contrib)) {
                    KzShdRec shd; shd.d = mkf4(es.wi.x, es.wi.y, es.wi.z, es.dist - eps); shd.pending = mkf4(contrib.x, contrib.y, contrib.z, eps);
                    st.c[slot].shd = shd;
                    flags |= KZ_SHADE_SHADOW;
                }
            }
        }
    } else if (sc.n_light_meshes > 0) {
        const uint32_t nl = (uint32_t)sc.n_light_meshes;
        const float u_tri = kz_next1d(sc, sm);
        const float u_b1 = kz_next1d(sc, sm);
        const float u_b2 = kz_next1d(sc, sm);
        const KzEmitterSample es = kz_sample_emitter(sc, its.p, rnd, u_tri, u_b1, u_b2);
        const kz3 lwi = es.wi;
        const float dist = es.dist, lpdf = es.pdf;
        if (lpdf > 0.f && !isnan(lpdf) && !isinf(lpdf)) {
            const kz_light_desc l = sc.lights[es.light];
            /* eval: cosTheta > 0 is implied by lpdf > 0 */
            kz3 Ls = mk3(l.radiance[0], l.radiance[1], l.radiance[2]) / lpdf;
            Ls = Ls / (1.f / (float)nl);
            kz3 f; float bsdfPdf;
            bsdf_eval_pdf(bc, its, wiLocal, to_local(its.sh, lwi), &f, &bsdfPdf);
            const float lightWeight = power_heuristic(lpdf, bsdfPdf);
            const kz3 contrib = throughput * Ls * f * lightWeight;
            if (!iszero(contrib)) {
                KzShdRec shd; shd.d = mkf4(lwi.x, lwi.y, lwi.z, dist - eps); shd.pending = mkf4(contrib.x, contrib.y, contrib.z, eps);
                st.c[slot].shd = shd;            /* origin: A.ray.o, written below */
                flags |= KZ_SHADE_SHADOW;
            }
        }
    }

    /* ---- regularisation, integrator.cpp:299-301 ---- */
    if (I.regularization) its.acc_rough += bsdf_regularize(bc) * I.accumulated_roughness;

    /* ---- BSDF sampling, integrator.cpp:304-314 ---- */
    KZ_DRAW_BSDF_SAMPLES(sc, sm, s1, s2);
    kz3 wo; float bsdfPdf, sampledEta; int measure;
    const kz3 weight = bsdf_sample(bc, its, wiLocal, s1, s2, &wo, &bsdfPdf, &measure, &sampledEta);
    throughput *= weight;
    eta *= sampledEta;
    if (measure == KZ_MEASURE_DISCRETE) bsdfPdf = -1.f;      /* flag for the next vertex: bsdfWeight = 1 (integrator.cpp:329-331) */
    KzBlockB B; B.rad.thr = mkf4(throughput.x, throughput.y, throughput.z, eta); B.rad.L = mkf4(L.x, L.y, L.z, bsdfPdf); B.smp = kz_sampler_save(sm, its.acc_rough);
    st.b[slot] = B;
    if (iszero(throughput)) {                /* dead path: every later term is multiplied by 0 */
        if (flags) st.a[slot].ray.o = mkf4(its.p.x, its.p.y, its.p.z, eps);
        return flags;
    }
    const kz3 wow = to_world(its.sh, wo);
    KzRayRec ray; ray.o = mkf4(its.p.x, its.p.y, its.p.z, eps); ray.d = mkf4(wow.x, wow.y, wow.z, KZ_INF);
    st.a[slot].ray = ray;
    return flags | KZ_SHADE_CONTINUE;
}

/* ---- the other integrators (SURVEY 8f-3): normals / ao / whitted / path_mats, integrator.cpp:11-181 -------------------- */
KZ_HD kz3 square_to_uniform_hemisphere(kz2 s) {            /* warp.cpp:68-79 */
    const float z = s.x, tmp = sqrtf(1.0f - z * z), phi = 2.0f * KZ_PI * s.y;
    return mk3(cosf(phi) * tmp, sinf(phi) * tmp, z);
}
/* One loop iteration of the selected integrator; thr = running weight, L = accumulated colour.  Every hit (and miss) goes
 * through this routine: these integrators are not material sorted. */
KZ_HD_NOINLINE uint32_t kz_shade_alt_item(const KzScene &sc, const KzPathState &st, uint32_t slot, int bounce, KzCounters &cnt) {
    const int type = sc.integrator.type;
    const KzBlockA A = st.a[slot];
    const KzF4 ro = A.ray.o, rd = A.ray.d;
    const kz3 rayO = mk3(ro.x, ro.y, ro.z), rayD = mk3(rd.x, rd.y, rd.z);
    KzHit h; h.t = A.hit.t; h.u = A.hit.u; h.v = A.hit.v; h.prim = A.hit.prim; h.geom = A.hit.geom;
    if (h.geom == KZ_INVALID_ID) return 0u;                /* every one of them returns what it has on a miss */
    const KzRadRec rad = st.b[slot].rad;
    KzF4 thr4 = rad.thr, L4 = rad.L;
    kz3 weight = mk3(thr4.x, thr4.y, thr4.z), L = mk3(L4.x, L4.y, L4.z);
    KzIts its; its.acc_rough = 0.f;
    fill_intersection(sc, h, its, mk3(0.f));
    const KzMeshRec mesh = sc.meshes[its.mesh];
    if (type == KZ_INTEGRATOR_NORMALS) {                   /* integrator.cpp:19-29 */
        st.b[slot].rad.L = mkf4(fabsf(its.geo_n.x), fabsf(its.geo_n.y), fabsf(its.geo_n.z), 1.f);
        return 0u;
    }
    KzSampler sm;
    kz_sampler_load(sm, st.b[slot].smp);
    if (type == KZ_INTEGRATOR_AO) {                        /* integrator.cpp:43-62 */
        const kz3 sample = square_to_uniform_hemisphere(kz_next2d(sc, sm));
        kz3 point = to_world(its.sh, sample);
        const float cosTheta = dot(normalized(point), normalized(its.sh.n));
        const float v = (cosTheta / KZ_PI) / (0.5f * KZ_INV_PI);
        st.a[slot].ray.o = mkf4(its.p.x, its.p.y, its.p.z, KZ_EPSILON);
        KzShdRec shd; shd.d = mkf4(point.x, point.y, point.z, KZ_INF); shd.pending = mkf4(v, v, v, KZ_EPSILON);
        st.c[slot].shd = shd;
        return KZ_SHADE_SHADOW;
    }
    const kz3 wiLocal = to_local(its.sh, -rayD);
    kz3 Le = mk3(0.f);
    if (mesh.flags & KZ_MESH_IS_LIGHT) {
        const kz3 lwi = normalized(its.p - rayO);
        if (dot(its.sh.n, -lwi) > 0.f) { const kz_light_desc l = sc.lights[mesh.light]; Le = mk3(l.radiance[0], l.radiance[1], l.radiance[2]); }
    }
    uint32_t flags = 0u;
    if (type == KZ_INTEGRATOR_WHITTED) {                   /* integrator.cpp:80-128 with the recursion unrolled */
        const KzBsdfCtx bc = bsdf_ctx(sc, its);
        if (!bc.is_nmap && bc.leaf_type == KZ_BSDF_DIFFUSE) {            /* BSDF::isDiffuse(), bsdf.cpp:77 */
            L += weight * Le;
            const float rnd = kz_next1d(sc, sm);
            if (sc.n_light_meshes > 0) {
                const uint32_t nl = (uint32_t)sc.n_light_meshes;
                const float u_tri = kz_next1d(sc, sm);
                const float u_b1 = kz_next1d(sc, sm);
                const float u_b2 = kz_next1d(sc, sm);
                const KzEmitterSample es = kz_sample_emitter(sc, its.p, rnd, u_tri, u_b1, u_b2);
                const kz3 lwi = es.wi;
                const float dist = es.dist, lpdf = es.pdf;
                if (lpdf > 0.f && !isnan(lpdf) && !isinf(lpdf)) {
                    const kz_light_desc l = sc.lights[es.light];
                    const kz3 Ls = mk3(l.radiance[0], l.radiance[1], l.radiance[2]) / lpdf;
                    float cosTheta = to_local(its.sh, lwi).z;
                    if (cosTheta < 0.f) cosTheta = 0.f;
                    kz3 f; float pdf_unused;
                    bsdf_eval_pdf(bc, its, wiLocal, to_local(its.sh, lwi), &f, &pdf_unused);
                    const kz3 Lr = weight * (f * Ls * cosTheta) / (1.0f / (float)nl);
                    if (!iszero(Lr)) {
                        st.a[slot].ray.o = mkf4(its.p.x, its.p.y, its.p.z, 0.f);         /* Ray3f(ref, wi, 0, dist): light.cpp:24 */
                        KzShdRec shd; shd.d = mkf4(lwi.x, lwi.y, lwi.z, dist); shd.pending = mkf4(Lr.x, Lr.y, Lr.z, 0.f);
                        st.c[slot].shd = shd;
                        flags |= KZ_SHADE_SHADOW;
                    }
                }
            }
            st.b[slot].rad.L = mkf4(L.x, L.y, L.z, 1.f);
            return flags;
        }
        KZ_DRAW_BSDF_SAMPLES(sc, sm, s1, s2);
        kz3 wo; float p; int measure; float e;
        const kz3 refl = bsdf_sample(bc, its, wiLocal, s1, s2, &wo, &p, &measure, &e);
        if (!(kz_next1d(sc, sm) < 0.95f)) { st.b[slot].rad.L = mkf4(0.f, 0.f, 0.f, 1.f); return 0u; }      /* the whole recursion returns 0 */
        weight = weight * refl / 0.95f;
        st.b[slot].smp = kz_sampler_save(sm, 0.f);
        st.b[slot].rad.thr = mkf4(weight.x, weight.y, weight.z, 1.f);
        if (iszero(weight) || bounce >= 4095) { st.b[slot].rad.L = mkf4(0.f, 0.f, 0.f, 1.f); return 0u; }
        const kz3 wow = to_world(its.sh, wo);
        KzRayRec ray; ray.o = mkf4(its.p.x, its.p.y, its.p.z, KZ_EPSILON); ray.d = mkf4(wow.x, wow.y, wow.z, KZ_INF);
        st.a[slot].ray = ray;
        return KZ_SHADE_CONTINUE;
    }
    /* path_mats, integrator.cpp:142-173 */
    L += weight * Le;
    st.b[slot].rad.L = mkf4(L.x, L.y, L.z, 1.f);
    const float probability = fminf(weight.x, 0.95f);
    if (kz_next1d(sc, sm) >= probability) return 0u;
    weight = weight / probability;
    cnt.vertices += 1;
    const KzBsdfCtx bc = bsdf_ctx(sc, its);
    KZ_DRAW_BSDF_SAMPLES(sc, sm, s1, s2);
    kz3 wo; float p; int measure; float e;
    const kz3 f = bsdf_sample(bc, its, wiLocal, s1, s2, &wo, &p, &measure, &e);
    weight *= f;
    st.b[slot].smp = kz_sampler_save(sm, 0.f);
    st.b[slot].rad.thr = mkf4(weight.x, weight.y, weight.z, 1.f);
    if (iszero(weight) || bounce >= 4095) return 0u;
    const kz3 wow = to_world(its.sh, wo);
    KzRayRec ray; ray.o = mkf4(its.p.x, its.p.y, its.p.z, KZ_EPSILON); ray.d = mkf4(wow.x, wow.y, wow.z, KZ_INF);
    st.a[slot].ray = ray;
    return KZ_SHADE_CONTINUE;
}

/* ---- shadow -------------------------------------------------------------------------------- */
/* integrator.cpp:259-278; returns true when occluded; *segments = closest-hit queries issued */
KZ_HD bool kz_occluded_walk(const KzScene &sc, const KzStackRef &stk, kz3 o, kz3 d, float tmin, float tmax, float eps, int *segments) {
    int seg = 0;
    bool occluded = false;
    for (;;) {
        ++seg;
        const KzHit h = kz_trace(sc, stk, o.x, o.y, o.z, d.x, d.y, d.z, tmin, tmax, false);
        if (h.geom == KZ_INVALID_ID) break;
        const uint32_t fl = sc.meshes[h.geom].flags;
        if (!(fl & KZ_MESH_IS_LIGHT) || (fl & KZ_MESH_LIGHT_VISIBLE) || sc.integrator.type != KZ_INTEGRATOR_PATH_MIS) { occluded = true; break; }
        o = o + d * (h.t + eps);
        tmin = eps;
        tmax = tmax - h.t;
        if (seg > 4096) break;
    }
    *segments = seg;
    return occluded;
}
KZ_HD void kz_shadow_item(const KzScene &sc, const KzStackRef &stk, const KzPathState &st, uint32_t slot, KzCounters &cnt) {
    const KzF4 so = st.a[slot].ray.o;
    const KzShdRec shd = st.c[slot].shd;
    int seg;
    const bool occ = kz_occluded_walk(sc, stk, mk3(so.x, so.y, so.z), mk3(shd.d.x, shd.d.y, shd.d.z), shd.pending.w, shd.d.w, sc.integrator.trace_bias, &seg);
    cnt.rays_shadow += (unsigned long long)seg;
    if (!occ) {
        KzF4 L = st.b[slot].rad.L;
        L.x += shd.pending.x; L.y += shd.pending.y; L.z += shd.pending.z;
        st.b[slot].rad.L = L;
    }
}

/* ---- accumulate ---------------------------------------------------------------------------- */
#if KZ_DEVICE_CODE
#define KZ_FRAME_ADD(ptr, vr, vg, vb, vw) atomicAdd(reinterpret_cast<float4 *>(ptr), make_float4(vr, vg, vb, vw))
#else
#define KZ_FRAME_ADD(ptr, vr, vg, vb, vw) do { (ptr)->x += (vr); (ptr)->y += (vg); (ptr)->z += (vb); (ptr)->w += (vw); } while (0)
#endif
/* ImageBlock::put on the whole bordered frame, block.cpp:56-85 */
/* `table`: the 33-entry filter table (the kernel reads it from a shared-memory copy: a dynamically indexed kernel parameter
 * serialises divergent lanes in the constant cache). */
/* What one path puts on the film: its value, its sample position and the texel rectangle of its filter footprint, all in the
 * coordinates of the bordered frame (block.cpp:56-76).  False if the value is invalid (block.cpp:58-62). */
struct KzSplat { kz3 value; float px, py; int x0, y0, x1, y1; int ipx, ipy; };
KZ_HD bool kz_splat_of(const KzScene &sc, const KzPathState &st, uint32_t slot, KzSplat &sp) {
    const KzF4 L = st.b[slot].rad.L;
    sp.value = mk3(L.x, L.y, L.z);
    if (!color_valid(sp.value)) return false;
    /* the pixel sample position is not carried with the path: the samplers are addressable by (pixel, sample index), so it is
     * drawn again exactly as in raygen (renderer.cpp:25-26) */
    const KzSmpRec smp = st.b[slot].smp;
    KzSampler sm;
    sp.ipx = (int32_t)(smp.pix & 0xFFFFu); sp.ipy = (int32_t)(smp.pix >> 16);
    kz_sampler_start(sc, sm, sp.ipx, sp.ipy, smp.sidx);
    const kz2 jitter = kz_next_pixel2d(sc, sm);
    const int b = sc.border, cols = sc.camera.width + 2 * b, rows = sc.camera.height + 2 * b;
    const float radius = sc.filter.radius;
    sp.px = ((float)sp.ipx + jitter.x) - 0.5f - (float)(0 - b); sp.py = ((float)sp.ipy + jitter.y) - 0.5f - (float)(0 - b);
    int x0 = (int)ceilf(sp.px - radius), y0 = (int)ceilf(sp.py - radius);
    int x1 = (int)floorf(sp.px + radius), y1 = (int)floorf(sp.py + radius);
    sp.x0 = x0 < 0 ? 0 : x0; sp.y0 = y0 < 0 ? 0 : y0;
    sp.x1 = x1 > cols - 1 ? cols - 1 : x1; sp.y1 = y1 > rows - 1 ? rows - 1 : y1;
    return true;
}

KZ_HD void kz_accumulate_item(const KzScene &sc, const KzPathState &st, uint32_t slot, KzF4 *frame, const float *table) {
    KzSplat sp;
    if (!kz_splat_of(sc, st, slot, sp)) return;
    const kz3 value = sp.value;
    const float px = sp.px, py = sp.py;
    const int x0 = sp.x0, y0 = sp.y0, x1 = sp.x1, y1 = sp.y1;
    const int cols = sc.camera.width + 2 * sc.border;
    const float lookup = 32 / sc.filter.radius;
    for (int y = y0; y <= y1; ++y) {
        const float wy = table[(int)(fabsf((float)y - py) * lookup)];
        for (int x = x0; x <= x1; ++x) {
            const float wx = table[(int)(fabsf((float)x - px) * lookup)];
            KzF4 *p = frame + ((size_t)y * cols + x);
            KZ_FRAME_ADD(p, value.x * wx * wy, value.y * wx * wy, value.z * wx * wy, 1.0f * wx * wy);
        }
    }
}

#endif
