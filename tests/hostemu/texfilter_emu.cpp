/* tests/hostemu/texfilter_emu.cpp -- DEVELOPMENT/TEST HARNESS, NOT A PRODUCT PATH.
 *
 * emu.cpp (the device routines compiled for the host) plus texture filtering: the camera constants of kz_texlod.h as the host computes
 * them at upload, the footprint body the filtered shade kernels run, the level choice and trilinear lookup of kz_shade.h over a pyramid
 * given by the caller, the upload's decision and pyramid layout, and the footprint probe.  Built as its own library (texfilter_emu.py) so
 * that the CPU suite can check each against a numpy restatement.
 */
#include "emu.cpp"
#include "../../nano-kazen_b200/csrc/kz_texlod.h"

namespace {
/* KzTexLod <-> 19 floats: camera_from_world[12], ddx[3], ddy[3], spp_scale */
void lod_out(const KzTexLod &l, float *o) {
    memcpy(o, l.camera_from_world, 48); memcpy(o + 12, l.ddx, 12); memcpy(o + 15, l.ddy, 12); o[18] = l.spp_scale;
}
KzTexLod lod_in(const float *o) {
    KzTexLod l;
    memcpy(l.camera_from_world, o, 48); memcpy(l.ddx, o + 12, 12); memcpy(l.ddy, o + 15, 12); l.spp_scale = o[18];
    return l;
}
kz3 v3(const float *p) { return mk3(p[0], p[1], p[2]); }
/* a one-image scene over the caller's pyramid (level 0 then levels 1 .. n_levels, float4 texels) */
struct OneImage {
    KzImageRec rec;
    KzScene sc;
    OneImage(int w, int h, int n_levels, const float *texels4) {
        rec.width = w; rec.height = h; rec.texel_offset = 0; rec.n_levels = n_levels;
        memset(&sc, 0, sizeof(sc));
        sc.images = &rec; sc.texels = reinterpret_cast<const KzF4 *>(texels4);
    }
};
}  // namespace

extern "C" {

/* kz_tex_lod of a camera and sample count (19 floats) */
int kztf_lod(const kz_camera_desc *c, uint32_t sample_count, float *out19) {
    lod_out(kz_tex_lod(*c, sample_count), out19);
    return KZ_OK;
}

/* kz_uv_footprint per case: 56 floats = lod[19], camera_to_world[16], p[3], n[3], p0[3], p1[3], p2[3], uv0[2], uv1[2], uv2[2]
 * -> du/dx, dv/dx, du/dy, dv/dy */
int kztf_footprint(const float *cases, size_t n, float *out4) {
    pfor(n, [&](size_t b, size_t e) {
        for (size_t i = b; i < e; ++i) {
            const float *c = cases + 56 * i;
            const float *g = c + 35;
            const KzUvDiff d = kz_uv_footprint(lod_in(c), c + 19, v3(g), v3(g + 3), v3(g + 6), v3(g + 9), v3(g + 12), mk2(g[15], g[16]), mk2(g[17], g[18]),
                                               mk2(g[19], g[20]));
            float *o = out4 + 4 * i;
            o[0] = d.dudx; o[1] = d.dvdx; o[2] = d.dudy; o[3] = d.dvdy;
        }
    });
    return KZ_OK;
}

/* kz_tex_lambda of a w x h image per (ds/dx, dt/dx, ds/dy, dt/dy) */
int kztf_lambda(int w, int h, const float *dst4, size_t n, float *out) {
    KzImageRec r; r.width = w; r.height = h; r.texel_offset = 0; r.n_levels = 0;
    for (size_t i = 0; i < n; ++i) out[i] = kz_tex_lambda(r, dst4[4 * i], dst4[4 * i + 1], dst4[4 * i + 2], dst4[4 * i + 3]);
    return KZ_OK;
}

/* kz_image_filtered at (s, t, lambda) per item, over the caller's pyramid */
int kztf_filtered(int w, int h, int n_levels, const float *texels4, const float *st, const float *lambda, size_t n, float *rgb) {
    OneImage im(w, h, n_levels, texels4);
    for (size_t i = 0; i < n; ++i) {
        const kz3 c = kz_image_filtered(im.sc, 0, st[2 * i], st[2 * i + 1], lambda[i]);
        rgb[3 * i] = c.x; rgb[3 * i + 1] = c.y; rgb[3 * i + 2] = c.z;
    }
    return KZ_OK;
}
/* kz_image_bicubic at `level` per (s, t), over the caller's pyramid */
int kztf_bicubic(int w, int h, int n_levels, const float *texels4, const float *st, int level, size_t n, float *rgb) {
    OneImage im(w, h, n_levels, texels4);
    for (size_t i = 0; i < n; ++i) {
        const kz3 c = kz_image_bicubic(im.sc, 0, st[2 * i], st[2 * i + 1], level);
        rgb[3 * i] = c.x; rgb[3 * i + 1] = c.y; rgb[3 * i + 2] = c.z;
    }
    return KZ_OK;
}
/* the filtered probe's body per (s, t, dst4) (k_image_lookup_filtered) */
int kztf_lookup_filtered(int w, int h, int n_levels, const float *texels4, const float *st, const float *dst4, size_t n, float *rgb) {
    OneImage im(w, h, n_levels, texels4);
    for (size_t i = 0; i < n; ++i) {
        const float *g = dst4 + 4 * i;
        const kz3 c = kz_image_filtered(im.sc, 0, st[2 * i], st[2 * i + 1], kz_tex_lambda(im.rec, g[0], g[1], g[2], g[3]));
        rgb[3 * i] = c.x; rgb[3 * i + 1] = c.y; rgb[3 * i + 2] = c.z;
    }
    return KZ_OK;
}

/* kzgpu_scene_upload's decision and layout: *counts = filter_counts(); when it counts, KZ_ERR_INVALID (message in err) if the pyramids do
 * not fit, else *total = texels of all levels and levels[i] = image i's n_levels.  Image arrays are never read (flatten without geometry). */
int kztf_layout(const kz_scene_desc *d, int *counts, uint64_t *total, int32_t *levels, char *err, size_t err_len) {
    KzHostScene hs;
    err[0] = 0;
    if (!hs.flatten(d, false)) { snprintf(err, err_len, "%s", hs.error.c_str()); return KZ_ERR_INVALID; }
    *counts = hs.filter_counts();
    if (*counts && !hs.mip_layout()) { snprintf(err, err_len, "%s", hs.error.c_str()); return KZ_ERR_INVALID; }
    *total = hs.total_texels;
    for (size_t i = 0; i < hs.images.size(); ++i) levels[i] = hs.images[i].n_levels;
    return KZ_OK;
}

/* kzgpu_texture_footprint_dump's layout (k_texture_footprint_dump) with the camera constants of the uploaded camera */
int kztf_footprint_dump(kzemu *e, const kz_ray *rays, size_t n, float *out8) {
    const KzScene &sc = e->hs.sc;
    const KzTexLod lod = kz_tex_lod(sc.camera, sc.sample_count);
    pfor(n, [&](size_t b, size_t en) {
        KzStackRef stk;
        for (size_t i = b; i < en; ++i) {
            const kz_ray &r = rays[i];
            const KzHit h = kz_trace(sc, stk, r.o[0], r.o[1], r.o[2], r.d[0], r.d[1], r.d[2], r.tmin, r.tmax, false);
            float *o = out8 + 8 * i;
            for (int k = 0; k < 8; ++k) o[k] = 0.f;
            o[0] = -1.f;
            if (h.geom == KZ_INVALID_ID) continue;
            KzIts its; its.acc_rough = 0.f;
            fill_intersection(sc, h, its, mk3(0.f));
            const KzUvDiff duv = kz_its_footprint(sc, lod, h, its);
            o[0] = (float)its.mesh; o[1] = its.uv.x; o[2] = its.uv.y;
            o[3] = duv.dudx; o[4] = duv.dvdx; o[5] = duv.dudy; o[6] = duv.dvdy;
        }
    });
    return KZ_OK;
}

}  // extern "C"
