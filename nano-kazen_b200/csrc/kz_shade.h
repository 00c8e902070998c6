/* kz_shade.h -- device shading library: textures, kiss / diffuse / normalmap BSDFs, area
 * lights, Mesh::sample, post-intersection.  References (nano-kazen):
 *   texture.cpp:10-270, bsdf.cpp:20-92,281-417,1157-1418, ggx_brdf.h:15-170, light.cpp:7-66,
 *   mesh.cpp:108-133, dpdf.h:99-104, accel.cpp:113-236, scene.cpp:54-79, warp.cpp:41-50,85-115.
 * Float math here may be contracted to FMA by nvcc (image parity is statistical, SURVEY
 * Appendix A 15a); sampler floats and hit t are produced elsewhere with exact rounding. */
#ifndef KZ_SHADE_H
#define KZ_SHADE_H
#include "kz_sampler.h"
#include "kz_traverse.h"

#define KZ_MEASURE_UNKNOWN 0
#define KZ_MEASURE_SOLID_ANGLE 1
#define KZ_MEASURE_DISCRETE 2

/* mesh.h:18-56 (subset that the hot path reads) */
struct KzIts {
    kz3 p;
    kz2 uv;
    KzFrame sh;
    kz3 geo_n;
    kz3 dpdu;
    int32_t mesh;
    float acc_rough;
};

/* ---- warps ---------------------------------------------------------------------------------- */
KZ_HD kz2 square_to_uniform_disk(kz2 s) {
    float r = sqrtf(s.x);
    float a = 2.0f * KZ_PI * s.y;
    return mk2(cosf(a) * r, sinf(a) * r);
}
KZ_HD kz3 square_to_cosine_hemisphere(kz2 s) {
    float r1 = 2.0f * s.x - 1.0f, r2 = 2.0f * s.y - 1.0f;
    float phi, r;
    if (r1 == 0 && r2 == 0) { r = phi = 0; }
    else if (r1 * r1 > r2 * r2) { r = r1; phi = (KZ_PI / 4.0f) * (r2 / r1); }
    else { r = r2; phi = (KZ_PI / 2.0f) - (r1 / r2) * (KZ_PI / 4.0f); }
    float px = r * cosf(phi), py = r * sinf(phi);
    float z = sqrtf(1.0f - px * px - py * py);
    if (z == 0) z = 1e-10f;
    return mk3(px, py, z);
}

/* ---- textures -------------------------------------------------------------------------------- */
KZ_HD int kz_wrapi(int i, int n) { int r = i % n; return r < 0 ? r + n : r; }
KZ_HD void kz_bspline_weights(float f, float w[4]) {
    float one_f = 1.0f - f;
    w[0] = (one_f * one_f * one_f) / 6.0f;
    w[1] = 2.0f / 3.0f - 0.5f * f * f * (2.0f - f);
    w[2] = 2.0f / 3.0f - 0.5f * one_f * one_f * (2.0f - one_f);
    w[3] = (f * f * f) / 6.0f;
}
/* Mip pyramid: level l (max(1,w>>l) x max(1,h>>l) float4 texels) follows level l-1, built on the GPU by 2x2 box filtering
 * (k_mip_level).  kazen calls OIIO with zero derivatives (texture.cpp:52-57), which selects the finest level, so the reference
 * render path always passes level 0.  With texture filtering (kz_integrator_desc::texture_filtering) every image's pyramid is
 * resident from the upload on and uv-mode lookups pick their level from the vertex's footprint (kz_image_filtered). */
KZ_HD void kz_mip_level(const KzImageRec &im, int level, int &w, int &h, size_t &offset) {
    w = im.width; h = im.height; offset = im.texel_offset;
    if (level > im.n_levels) level = im.n_levels;
    for (int l = 0; l < level; ++l) {
        offset += (size_t)w * (size_t)h;
        w = w > 1 ? w >> 1 : 1; h = h > 1 ? h >> 1 : 1;
    }
}
/* periodic wrap, bicubic B-spline (OIIO's default interpolation when magnifying) */
KZ_HD_NOINLINE kz3 kz_image_bicubic(const KzScene &sc, int image, float s, float t, int level = 0) {
    const KzImageRec im = sc.images[image];
    int w = im.width, h = im.height; size_t off = im.texel_offset;
    if (level > 0) kz_mip_level(im, level, w, h, off);
    float x = s * w - 0.5f, y = t * h - 0.5f;
    float fx = floorf(x), fy = floorf(y);
    int ix = (int)fx, iy = (int)fy;
    float wx[4], wy[4];
    kz_bspline_weights(x - fx, wx);
    kz_bspline_weights(y - fy, wy);
    kz3 acc = mk3(0.f);
    const KzF4 *base = sc.texels + off;
    for (int j = 0; j < 4; ++j) {
        int yy = kz_wrapi(iy - 1 + j, h);
        kz3 row = mk3(0.f);
        for (int i = 0; i < 4; ++i) {
            int xx = kz_wrapi(ix - 1 + i, w);
            const KzF4 p = base[(size_t)yy * w + xx];
            row += mk3(p.x, p.y, p.z) * wx[i];
        }
        acc += row * wy[j];
    }
    return acc;
}

/* Footprint of a shading vertex in texture space: uv derivatives per pixel step in x and y (kz_texlod.h computes them). */
struct KzUvDiff { float dudx, dvdx, dudy, dvdy; };

/* pbrt-v4's trilinear level (MIPMap::Filter) of an isotropic lookup whose st derivatives are dst = (ds/dx, dt/dx, ds/dy, dt/dy):
 * log2 of twice the longest footprint axis in texels (exact for square power-of-two images, the longer side's texels otherwise). */
KZ_HD float kz_tex_lambda(const KzImageRec &im, float dsdx, float dtdx, float dsdy, float dtdy) {
    const float w = (float)im.width, h = (float)im.height;
    const float width = 2.0f * fmaxf(fmaxf(fabsf(dsdx) * w, fabsf(dtdx) * h), fmaxf(fabsf(dsdy) * w, fabsf(dtdy) * h));
    return log2f(fmaxf(width, 1e-8f));
}
/* Trilinear lookup at level lambda: lambda <= 0 is the reference's level-0 lookup itself, lambda >= n_levels the top level, and in
 * between the lerp of the bicubic lookups of the two levels around it (bicubic per level, so that a magnified texture is the reference). */
KZ_HD kz3 kz_image_filtered(const KzScene &sc, int image, float s, float t, float lambda) {
    if (!(lambda > 0.f)) return kz_image_bicubic(sc, image, s, t);
    const int top = sc.images[image].n_levels;
    if (lambda >= (float)top) return kz_image_bicubic(sc, image, s, t, top);
    const int l = (int)floorf(lambda);
    const float f = lambda - (float)l;
    const kz3 a = kz_image_bicubic(sc, image, s, t, l), b = kz_image_bicubic(sc, image, s, t, l + 1);
    return (1.f - f) * a + f * b;
}

/* Expression trees are tiny (depth <= 3 in every kazen scene).  They are evaluated post-order
 * with an explicit frame stack of bounded depth: no recursion (no device call stack growth) and
 * no template expansion (a blend has three children; inlining the tree is exponential).
 * dir_mode: Texture::eval(dir) (texture.cpp:66-81,121-126) instead of eval(uv).
 * FILT: uv-mode image lookups are filtered by the footprint `duv` (kz_image_filtered); without it every lookup reads level 0. */
#define KZ_TEX_MAX_DEPTH 4
template <bool FILT>
KZ_HD kz3 kz_tex_eval_body(const KzScene &sc, int root, kz2 uv_, kz3 d, bool dir_mode, const KzUvDiff &duv) {
    int node[KZ_TEX_MAX_DEPTH], next[KZ_TEX_MAX_DEPTH];
    kz3 val[KZ_TEX_MAX_DEPTH][3];
    int sp = 0;
    node[0] = root; next[0] = 0;
    for (;;) {
        const kz_texture_desc t = sc.textures[node[sp]];
        int nchild = t.type == KZ_TEX_BLEND ? 3 : ((t.type == KZ_TEX_BACKGROUND || t.type == KZ_TEX_COLORRAMP) ? 1 : 0);
        if (dir_mode && t.type != KZ_TEX_BACKGROUND) nchild = 0;     /* only background forwards eval(dir) */
        if (next[sp] < nchild) {
            const int k = next[sp];
            const int c = t.child[k];
            if (c < 0 || sp + 1 == KZ_TEX_MAX_DEPTH) {
                /* blend defaults, texture.cpp:215-217; a missing unary child evaluates to 0 below */
                val[sp][k] = (t.type == KZ_TEX_BLEND && c < 0) ? (k == 0 ? mk3(0.5f) : (k == 1 ? mk3(0.f) : mk3(1.f))) : mk3(0.f);
                next[sp] = k + 1;
            } else {
                ++sp; node[sp] = c; next[sp] = 0;
            }
            continue;
        }
        kz3 r = mk3(0.f);
        switch (t.type) {
            case KZ_TEX_CONSTANT: r = mk3(t.color[0], t.color[1], t.color[2]); break;
            case KZ_TEX_IMAGE:
                if (dir_mode) {
                    float s = atan2f(-d.x, d.z) / (2.0f * KZ_PI) + 0.5f;
                    float tt = 0.5f - atan2f(d.y, hypotf(d.z, -d.x)) / KZ_PI;
                    if (isnan(s)) s = 0.0f;
                    if (isnan(tt)) tt = 0.0f;
                    r = kz_image_bicubic(sc, t.image, s, tt);
                } else {
                    if (FILT)      /* s = u * scale, t = (1 - v) * scale: ds = scale * du, dt = -scale * dv */
                        r = kz_image_filtered(sc, t.image, uv_.x * t.scale, (1.0f - uv_.y) * t.scale,
                                              kz_tex_lambda(sc.images[t.image], t.scale * duv.dudx, -t.scale * duv.dvdx, t.scale * duv.dudy, -t.scale * duv.dvdy));
                    else
                        r = kz_image_bicubic(sc, t.image, uv_.x * t.scale, (1.0f - uv_.y) * t.scale);
                    if (t.srgb) r = mk3(srgb_to_linear1(r.x), srgb_to_linear1(r.y), srgb_to_linear1(r.z));
                }
                break;
            case KZ_TEX_BACKGROUND: r = t.child[0] >= 0 ? t.a * val[sp][0] : mk3(0.f); break;
            case KZ_TEX_COLORRAMP:
                if (!dir_mode && t.child[0] >= 0) {
                    const kz3 c = val[sp][0];
                    r = mk3(t.a + (t.b - t.a) * clampf(c.x, 0.f, 1.f), t.a + (t.b - t.a) * clampf(c.y, 0.f, 1.f), t.a + (t.b - t.a) * clampf(c.z, 0.f, 1.f));
                }
                break;
            case KZ_TEX_BLEND:
                if (!dir_mode) {
                    const kz3 mask = val[sp][0], in1 = val[sp][1], in2 = val[sp][2];
                    if (t.mode == KZ_BLEND_MIX) r = mk3(lerpf(mask.x, in1.x, in2.x), lerpf(mask.x, in1.y, in2.y), lerpf(mask.x, in1.z, in2.z));
                    else if (t.mode == KZ_BLEND_MULTIPLY) r = in1 * in2;
                }
                break;
            default: break;
        }
        if (sp == 0) return r;
        --sp;
        val[sp][next[sp]] = r;
        next[sp] += 1;
    }
}
KZ_HD_NOINLINE kz3 kz_tex_eval_tree(const KzScene &sc, int root, kz2 uv_, kz3 d, bool dir_mode) {
    return kz_tex_eval_body<false>(sc, root, uv_, d, dir_mode, KzUvDiff{0.f, 0.f, 0.f, 0.f});
}
KZ_HD_NOINLINE kz3 kz_tex_eval_tree(const KzScene &sc, int root, kz2 uv_, KzUvDiff duv) {     /* uv mode, filtered */
    return kz_tex_eval_body<true>(sc, root, uv_, mk3(0.f), false, duv);
}
template <bool FILT = false>
KZ_HD kz3 kz_tex_uv(const KzScene &sc, int node, kz2 uv, const KzUvDiff &duv = KzUvDiff{0.f, 0.f, 0.f, 0.f}) {
    const kz_texture_desc *t = sc.textures + node;
    if (t->type == KZ_TEX_CONSTANT) return mk3(t->color[0], t->color[1], t->color[2]);     /* the common case */
    if (FILT) return kz_tex_eval_tree(sc, node, uv, duv);
    return kz_tex_eval_tree(sc, node, uv, mk3(0.f), false);
}
KZ_HD kz3 kz_background(const KzScene &sc, kz3 d) {   /* scene.cpp:54-79 */
    if (sc.background < 0) return mk3(0.f);
    if (isnan3(d)) return mk3(0.f);
    return kz_tex_eval_tree(sc, sc.background, mk2(0.f, 0.f), d, true);
}

/* ---- GGX helpers (ggx_brdf.h) ------------------------------------------------------------ */
KZ_HD kz2 roughness_to_alpha(float roughness, float anisotropy) {
    float alpha = fmaxf(0.001f, sqr(roughness));
    return mk2(alpha * (1.0f + anisotropy), alpha * (1.0f - anisotropy));
}
KZ_HD float ggx_lambda(kz3 v, kz2 a) {
    float squared = (sqr(a.x) * sqr(v.x) + sqr(a.y) * sqr(v.y)) / sqr(v.z);
    return (-1.0f + sqrtf(1.0f + squared)) * 0.5f;
}
KZ_HD float smith_g1(kz3 V, kz3 H, kz2 a) { return dot(V, H) <= 0.0f ? 0.0f : 1.0f / (1.0f + ggx_lambda(V, a)); }
KZ_HD float smith_g2(kz3 V, kz3 L, kz3 H, kz2 a) {
    if (dot(V, H) <= 0.0f || dot(L, H) < 0.0f) return 0.0f;
    return 1.0f / (1.0f + ggx_lambda(V, a) + ggx_lambda(L, a));
}
KZ_HD float ggx_ndf(kz3 H, kz2 a) {
    float ellipse = sqr(H.x) / sqr(a.x) + sqr(H.y) / sqr(a.y) + sqr(H.z);
    return 1.0f / (KZ_PI * a.x * a.y * sqr(ellipse));
}
KZ_HD float ggx_vndf(kz3 V, kz3 H, kz2 a) {
    float VDotH = dot(V, H);
    if (VDotH <= 0.0f) return 0.0f;
    return ggx_ndf(H, a) * smith_g1(V, H, a) * VDotH / V.z;
}
KZ_HD kz3 sample_ggx_vndf(kz3 V, kz2 a, kz2 rnd) {
    kz3 Vh = normalized(mk3(a.x * V.x, a.y * V.y, V.z));
    float lensq = Vh.x * Vh.x + Vh.y * Vh.y;
    kz3 T1 = lensq > 0.0f ? mk3(-Vh.y, Vh.x, 0.0f) / sqrtf(lensq) : mk3(1.0f, 0.0f, 0.0f);
    kz3 T2 = normalized(cross(Vh, T1));
    float r = sqrtf(rnd.x);
    float phi = 2.0f * KZ_PI * rnd.y;
    float t1 = r * cosf(phi);
    float t2 = r * sinf(phi);
    float s = 0.5f * (1.0f + Vh.z);
    t2 = (1.0f - s) * sqrtf(1.0f - t1 * t1) + s * t2;
    kz3 Nh = t1 * T1 + t2 * T2 + sqrtf(fmaxf(0.0f, 1.0f - t1 * t1 - t2 * t2)) * Vh;
    return normalized(mk3(a.x * Nh.x, a.y * Nh.y, fmaxf(1e-6f, Nh.z)));
}
KZ_HD kz3 ggx_smith_brdf(kz3 V, kz3 L, kz3 f0, float roughness, float anisotropy) {
    if (V.z * L.z < 0.0f) return mk3(0.0f);
    kz2 a = roughness_to_alpha(roughness, anisotropy);
    kz3 H = normalized(V + L);
    float D = ggx_ndf(H, a);
    float G = smith_g2(V, L, H, a);
    float w = powf(1.0f - dot(V, H), 5.0f);
    kz3 F = f0 * 1.0f + (mk3(1.f) - f0) * w;
    float denom = 4.0f * fabsf(V.z) * fabsf(L.z);
    return (D * G) * F / denom;
}

/* ---- BSDF query record (bsdf.h:17-53), minimal ------------------------------------------- */
struct KzBRec {
    kz3 wi, wo;
    kz2 uv;
    float acc_rough;     /* bRec.its.accumulatedRoughness */
    float eta;
    int measure;
};

KZ_HD float schlick_weight(float x) { x = clampf(1.f - x, 0.f, 1.f); float x2 = x * x; return x2 * x2 * x; }
KZ_HD kz3 lerp_color(kz3 c1, kz3 c2, float t) { return (1.f - t) * c1 + t * c2; }

/* Texture fetches of one kiss lookup, shared by eval/pdf/sample of the same vertex. */
struct KzKissParams { kz3 base; float metallic, roughness_raw; };
template <bool FILT = false>
KZ_HD KzKissParams kiss_params(const KzScene &sc, const kz_bsdf_desc &m, kz2 uv, const KzUvDiff &duv = KzUvDiff{0.f, 0.f, 0.f, 0.f}) {
    KzKissParams p;
    p.base = kz_tex_uv<FILT>(sc, m.base_color, uv, duv);
    p.metallic = kz_tex_uv<FILT>(sc, m.metallic, uv, duv).x;
    p.roughness_raw = kz_tex_uv<FILT>(sc, m.roughness, uv, duv).x;
    return p;
}
KZ_HD_NOINLINE kz3 kiss_eval(const kz_bsdf_desc &m, const KzKissParams &kp, const KzBRec &b) {   /* bsdf.cpp:1215-1267 */
    if (b.wi.z <= 0 || b.wo.z <= 0) return mk3(0.0f);
    kz3 V = b.wi, L = b.wo, H = normalized(V + L);
    kz3 Cdlin = kp.base;
    float metallic = kp.metallic;
    float roughness = fminf(1.f, kp.roughness_raw + b.acc_rough);
    float Cdlum = luminance(Cdlin);
    kz3 Ctint = Cdlum > 0.f ? Cdlin / Cdlum : mk3(1.f);
    kz3 Ctintmix = (0.08f * m.specular) * lerp_color(mk3(1.f), Ctint, m.specular_tint);
    kz3 Cspec0 = lerp_color(Ctintmix, Cdlin, metallic);
    float FL = schlick_weight(L.z), FV = schlick_weight(V.z), FH = schlick_weight(dot(L, H));
    float cosThetaD = dot(V, H);
    float Lambert = (1.f - 0.5f * FL) * (1.f - 0.5f * FV);
    float RR = 2.f * roughness * cosThetaD * cosThetaD;
    float retro = RR * (FL + FV + FL * FV * (RR - 1.f));
    kz3 Csheen = lerp_color(mk3(1.f), Ctint, m.sheen_tint);
    kz3 Fsheen = (FH * m.sheen) * Csheen;
    kz3 specTerm = ggx_smith_brdf(V, L, Cspec0, roughness, m.anisotropy);
    float ccR = lerpf(m.clearcoat_roughness, .01f, .3f);
    kz3 coatTerm = m.clearcoat != 0.f ? (0.25f * m.clearcoat) * ggx_smith_brdf(V, L, mk3(0.04f), ccR, m.anisotropy) : mk3(0.f);
    return ((1.f - metallic) * (Cdlin * KZ_INV_PI * (Lambert + retro) + Fsheen) + (specTerm + coatTerm)) * b.wo.z;
}
KZ_HD_NOINLINE float kiss_pdf(const kz_bsdf_desc &m, const KzKissParams &kp, const KzBRec &b) {   /* bsdf.cpp:1269-1299 */
    if (b.wi.z <= 0 || b.wo.z <= 0) return 0.0f;
    float diffuse = (1.f - kp.metallic) * 0.5f;
    float GTR2 = 1.f / (1.f + m.clearcoat);
    kz3 H = normalized(b.wi + b.wo);
    float jacobian = 4.0f * dot(b.wi, H);
    float roughness = fminf(1.f, kp.roughness_raw + b.acc_rough);
    kz2 alpha = roughness_to_alpha(roughness, m.anisotropy);
    float specPdf = ggx_vndf(b.wi, H, alpha) / jacobian;
    kz2 coatalpha = roughness_to_alpha(lerpf(m.clearcoat_roughness, .01f, .3f), 0.f);
    float coatPdf = ggx_vndf(b.wi, H, coatalpha) / jacobian;
    return diffuse * KZ_INV_PI * b.wo.z + (1.f - diffuse) * (GTR2 * specPdf + (1.f - GTR2) * coatPdf);
}
/* returns weight; *pdf_out = pdf(bRec) as the integrator queries it afterwards (integrator.cpp:314) */
KZ_HD_NOINLINE kz3 kiss_sample(const kz_bsdf_desc &m, const KzKissParams &kp, KzBRec &b, float sample1, kz2 sample2, float *pdf_out) { /* bsdf.cpp:1301-1371 */
    *pdf_out = 0.f;
    if (b.wi.z <= 0) return mk3(0.0f);
    b.measure = KZ_MEASURE_SOLID_ANGLE;
    b.eta = 1.0f;
    float diffuse = (1.f - kp.metallic) * 0.5f;
    if (sample1 < diffuse) {
        b.wo = square_to_cosine_hemisphere(sample2);
    } else {
        float sample = (sample1 - diffuse) / (1.f - diffuse);
        float GTR2 = 1.f / (1.f + m.clearcoat);
        kz2 alpha = sample < GTR2 ? roughness_to_alpha(kp.roughness_raw, m.anisotropy)      /* un-biased roughness, :1323 */
                                  : roughness_to_alpha(lerpf(m.clearcoat_roughness, 0.01f, .3f), 0.f);
        kz3 H = sample_ggx_vndf(b.wi, alpha, sample2);     /* flip is dead code: wi.z > 0 here */
        b.wo = normalized(reflect3(b.wi, H));
    }
    float pdf = kiss_pdf(m, kp, b);
    *pdf_out = pdf;
    if (b.wo.z <= 0 || pdf <= KZ_EPSILON || isnan3(b.wo)) return mk3(0.f);
    return kiss_eval(m, kp, b) / pdf;
}

/* ---- SURVEY 8(f)-1: dielectric, mirror, lambertian, ggx, roughconductor, roughplastic, roughdielectric ------------ */
KZ_HD float fresnel_ext_int(float cosThetaI, float extIOR, float intIOR) {                  /* common.cpp:447-476 */
    float etaI = extIOR, etaT = intIOR;
    if (extIOR == intIOR) return 0.0f;
    if (cosThetaI < 0.0f) { const float t = etaI; etaI = etaT; etaT = t; cosThetaI = -cosThetaI; }
    const float eta = etaI / etaT, sinThetaTSqr = eta * eta * (1 - cosThetaI * cosThetaI);
    if (sinThetaTSqr > 1.0f) return 1.0f;
    const float cosThetaT = sqrtf(1.0f - sinThetaTSqr);
    const float Rs = (etaI * cosThetaI - etaT * cosThetaT) / (etaI * cosThetaI + etaT * cosThetaT);
    const float Rp = (etaT * cosThetaI - etaI * cosThetaT) / (etaT * cosThetaI + etaI * cosThetaT);
    return (Rs * Rs + Rp * Rp) / 2.0f;
}
KZ_HD float fresnel_dielectric(float cosThetaI_, float eta, float &cosThetaT_) {            /* common.cpp:493-518 */
    const float scale = (cosThetaI_ > 0.f) ? 1 / eta : eta, cosThetaTSqr = 1 - (1 - cosThetaI_ * cosThetaI_) * (scale * scale);
    if (cosThetaTSqr <= 0.0f) { cosThetaT_ = 0.0f; return 1.0f; }
    const float cosThetaI = fabsf(cosThetaI_), cosThetaT = sqrtf(cosThetaTSqr);
    const float Rs = (cosThetaI - eta * cosThetaT) / (cosThetaI + eta * cosThetaT);
    const float Rp = (eta * cosThetaI - cosThetaT) / (eta * cosThetaI + cosThetaT);
    cosThetaT_ = (cosThetaI_ > 0) ? -cosThetaT : cosThetaT;
    return 0.5f * (Rs * Rs + Rp * Rp);
}
KZ_HD kz3 refract_dir(kz3 wi, kz3 n, float eta) {                                           /* common.cpp:525-534 */
    const float cosThetaI = dot(wi, n);
    if (cosThetaI < 0) eta = 1.0f / eta;
    const float cosThetaT2 = 1 - (1 - cosThetaI * cosThetaI) * (eta * eta);
    if (cosThetaT2 <= 0.0f) return mk3(0.0f);
    const float sign = cosThetaI >= 0.0f ? 1.0f : -1.0f;
    return n * (-cosThetaI * eta + sign * sqrtf(cosThetaT2)) + wi * eta;
}
KZ_HD float tan_theta(kz3 v) { const float t = 1 - v.z * v.z; return t <= 0.0f ? 0.0f : sqrtf(t) / v.z; }   /* frame.h:63-68 */
KZ_HD kz3 square_to_beckmann(kz2 s, float alpha) {                                          /* warp.cpp:121-125 */
    const float phi = 2 * KZ_PI * s.x;
    const float theta = atanf(alpha * sqrtf(logf(1 / (1 - s.y))));
    return mk3(sinf(theta) * cosf(phi), sinf(theta) * sinf(phi), cosf(theta));
}
KZ_HD float square_to_beckmann_pdf(kz3 m, float alpha) {                                    /* warp.cpp:127-130 */
    const float theta = acosf(m.z / norm(m));
    const bool ok = fabsf(norm(m) - 1) < KZ_EPSILON && m.z >= 0;
    return ok ? expf(-powf(tanf(theta), 2.f) / (alpha * alpha)) / (KZ_PI * alpha * alpha * powf(cosf(theta), 3.f)) : 0.f;
}
KZ_HD float beckmann_d(kz3 m, float alpha) {                                                /* bsdf.cpp:730-736 */
    const float temp = tan_theta(m) / alpha, ct = m.z, ct2 = ct * ct;
    return expf(-temp * temp) / (KZ_PI * alpha * alpha * ct2 * ct2);
}
KZ_HD float beckmann_g1(kz3 v, kz3 m, float alpha) {                                        /* bsdf.cpp:739-762 */
    if (dot(v, m) * v.z <= 0.0f) return 0.0f;
    const float tanTheta = fabsf(tan_theta(v));
    if (tanTheta == 0.0f) return 1.0f;
    const float a = 1.0f / (alpha * tanTheta);
    if (a >= 1.6f) return 1.0f;
    const float aSqr = a * a;
    return (3.535f * a + 2.181f * aSqr) / (1.0f + 2.276f * a + 2.577f * aSqr);
}
KZ_HD kz3 fresnel_cond(float c, kz3 eta, kz3 k) {                                           /* bsdf.cpp:718-727 */
    const kz3 tmp_f = eta * eta + k * k;
    const kz3 tmp = tmp_f * (c * c);
    const kz3 e2 = 2.f * eta * c;
    const kz3 Rparl2 = (tmp - e2 + mk3(1.f)) / (tmp + e2 + mk3(1.f));
    const kz3 Rperp2 = (tmp_f - e2 + mk3(c * c)) / (tmp_f + e2 + mk3(c * c));
    return (Rparl2 + Rperp2) * 0.5f;
}
KZ_HD float kd_max(const kz_bsdf_desc &m) { return fmaxf(m.albedo[0], fmaxf(m.albedo[1], m.albedo[2])); }

/* FILT: the base_color texture of lambertian / ggx is filtered by the vertex's footprint `duv` (extra_eval / extra_sample with it) */
template <bool FILT>
KZ_HD kz3 extra_eval_body(const KzScene &sc, const kz_bsdf_desc &m, const KzBRec &b, const KzUvDiff &duv) {
    const kz3 wi = b.wi, wo = b.wo;
    switch (m.type) {
        case KZ_BSDF_LAMBERTIAN:                                                             /* bsdf.cpp:211-221 */
            if (b.measure != KZ_MEASURE_SOLID_ANGLE || wi.z <= 0 || wo.z <= 0) return mk3(0.f);
            return kz_tex_uv<FILT>(sc, m.base_color, b.uv, duv) * KZ_INV_PI * wo.z;
        case KZ_BSDF_GGX:                                                                    /* bsdf.cpp:640-647 */
            if (wi.z <= 0 || wo.z <= 0) return mk3(0.f);
            return ggx_smith_brdf(wi, wo, kz_tex_uv<FILT>(sc, m.base_color, b.uv, duv), m.alpha, m.anisotropy) * wo.z;
        case KZ_BSDF_ROUGHCONDUCTOR: {                                                       /* bsdf.cpp:765-775 */
            if (wi.z <= 0 || wo.z <= 0) return mk3(0.f);
            const kz3 wh = normalized(wi + wo);
            const kz3 F = fresnel_cond(dot(wh, wo), mk3(m.eta[0], m.eta[1], m.eta[2]), mk3(m.k[0], m.k[1], m.k[2]));
            const float D = beckmann_d(wh, m.alpha);
            const float G = beckmann_g1(wi, wh, m.alpha) * beckmann_g1(wo, wh, m.alpha);
            return D * F * G / (4.f * wi.z);
        }
        case KZ_BSDF_ROUGHPLASTIC: {                                                         /* bsdf.cpp:881-893 */
            if (wi.z <= 0 || wo.z <= 0) return mk3(0.f);
            const kz3 kd = mk3(m.albedo[0], m.albedo[1], m.albedo[2]);
            const float ks = 1 - kd_max(m);
            const kz3 wh = normalized(wi + wo);
            const float D = beckmann_d(wh, m.alpha);
            const float F = fresnel_ext_int(dot(wh, wo), m.ext_ior, m.int_ior);
            const float G = beckmann_g1(wo, wh, m.alpha) * beckmann_g1(wi, wh, m.alpha);
            return kd * KZ_INV_PI * wo.z + mk3(ks * (D * F * G) / (4.f * wi.z));
        }
        case KZ_BSDF_ROUGHDIELECTRIC: {                                                      /* bsdf.cpp:969-1014 */
            if (wi.z == 0) return mk3(0.f);
            const float m_eta = m.int_ior / m.ext_ior, m_invEta = m.ext_ior / m.int_ior;
            const float cosThetaI = wi.z, cosThetaO = wo.z;
            const bool reflectS = cosThetaI * cosThetaO > 0.f;
            const float eta = cosThetaI > 0.f ? m_eta : m_invEta;
            kz3 wm = reflectS ? normalized(wi + wo) : normalized(wi + wo * eta);
            wm = wm * (wm.z > 0.f ? 1.f : -1.f);                                             /* math::sign */
            float ct;
            const float F = fresnel_dielectric(dot(wi, wm), m_eta, ct);
            const float D = beckmann_d(wm, m.alpha);
            const float G = beckmann_g1(wo, wm, m.alpha) * beckmann_g1(wi, wm, m.alpha);
            if (reflectS) return mk3((F * G * D) / (4.f * fabsf(cosThetaI)));
            const float denom = dot(wi, wm) + eta * dot(wo, wm);
            const float value = ((1 - F) * D * G * eta * eta * dot(wi, wm) * dot(wo, wm)) / (cosThetaI * sqr(denom));
            return mk3(fabsf(value));
        }
        default: return mk3(0.f);                                                            /* dielectric, mirror: discrete */
    }
}
KZ_HD_NOINLINE kz3 extra_eval(const KzScene &sc, const kz_bsdf_desc &m, const KzBRec &b) {
    return extra_eval_body<false>(sc, m, b, KzUvDiff{0.f, 0.f, 0.f, 0.f});
}
KZ_HD_NOINLINE kz3 extra_eval(const KzScene &sc, const kz_bsdf_desc &m, const KzBRec &b, KzUvDiff duv) {
    return extra_eval_body<true>(sc, m, b, duv);
}
KZ_HD_NOINLINE float extra_pdf(const kz_bsdf_desc &m, const KzBRec &b) {
    const kz3 wi = b.wi, wo = b.wo;
    switch (m.type) {
        case KZ_BSDF_LAMBERTIAN:                                                             /* bsdf.cpp:223-239 */
            if (b.measure != KZ_MEASURE_SOLID_ANGLE || wi.z <= 0 || wo.z <= 0) return 0.f;
            return KZ_INV_PI * wo.z;
        case KZ_BSDF_GGX: {                                                                  /* bsdf.cpp:649-657 */
            if (wi.z <= 0 || wo.z <= 0) return 0.f;
            const kz3 H = normalized(wi + wo);
            return ggx_vndf(wi, H, roughness_to_alpha(m.alpha, m.anisotropy)) / (4.0f * dot(wi, H));
        }
        case KZ_BSDF_ROUGHCONDUCTOR: {                                                       /* bsdf.cpp:778-785 */
            if (wi.z <= 0 || wo.z <= 0) return 0.f;
            const kz3 wh = normalized(wi + wo);
            return beckmann_d(wh, m.alpha) * wh.z * (1.f / (4.f * dot(wh, wo)));
        }
        case KZ_BSDF_ROUGHPLASTIC: {                                                         /* bsdf.cpp:895-903 */
            if (wi.z <= 0 || wo.z <= 0) return 0.f;
            const float ks = 1 - kd_max(m);
            const kz3 wh = normalized(wi + wo);
            const float Jh = 1.f / (4.f * fabsf(dot(wh, wo)));
            return ks * beckmann_d(wh, m.alpha) * wh.z * Jh + (1 - ks) * wo.z * KZ_INV_PI;
        }
        case KZ_BSDF_ROUGHDIELECTRIC: {                                                      /* bsdf.cpp:1016-1048 */
            const float m_eta = m.int_ior / m.ext_ior, m_invEta = m.ext_ior / m.int_ior;
            const float cosThetaI = wi.z, cosThetaO = wo.z;
            const bool reflectS = cosThetaI * cosThetaO > 0.f;
            const float eta = cosThetaI > 0.f ? m_eta : m_invEta;
            kz3 wm; float dwm_dwo;
            if (reflectS) { wm = normalized(wi + wo); dwm_dwo = 1.0f / (4.0f * dot(wo, wm)); }
            else {
                wm = normalized(wi + wo * eta);
                const float sqrtDenom = dot(wi, wm) + eta * dot(wo, wm);
                dwm_dwo = (eta * eta * dot(wo, wm)) / (sqrtDenom * sqrtDenom);
            }
            wm = wm * (wm.z > 0.f ? 1.f : -1.f);
            float ct;
            const float F = fresnel_dielectric(dot(wi, wm), m_eta, ct);
            float prob = beckmann_d(wm, m.alpha) * wm.z;
            prob *= reflectS ? F : (1 - F);
            return fabsf(prob * dwm_dwo);
        }
        default: return 0.f;
    }
}
/* returns the weight; *pdf_out = pdf(bRec) as the integrator queries it afterwards (integrator.cpp:314) */
template <bool FILT>
KZ_HD kz3 extra_sample_body(const KzScene &sc, const kz_bsdf_desc &m, KzBRec &b, float sample1, kz2 sample2, float *pdf_out, const KzUvDiff &duv) {
    *pdf_out = 0.f;
    kz3 w = mk3(0.f);
    switch (m.type) {
        case KZ_BSDF_DIELECTRIC: {                                                           /* bsdf.cpp:118-144 */
            b.measure = KZ_MEASURE_DISCRETE;
            const float fr = fresnel_ext_int(b.wi.z, m.ext_ior, m.int_ior);
            if (sample1 < fr) { b.wo = mk3(-b.wi.x, -b.wi.y, b.wi.z); b.eta = 1.f; return mk3(1.0f); }
            kz3 n = mk3(0.f, 0.f, 1.f);
            float factor = m.int_ior / m.ext_ior;
            if (b.wi.z < 0.f) { factor = m.ext_ior / m.int_ior; n.z = -1.0f; }
            b.wo = refract_dir(-b.wi, n, factor);
            b.eta = m.int_ior / m.ext_ior;
            return mk3(1.0f);
        }
        case KZ_BSDF_MIRROR:                                                                 /* bsdf.cpp:176-191 */
            if (b.wi.z <= 0) return mk3(0.f);
            b.wo = mk3(-b.wi.x, -b.wi.y, b.wi.z);
            b.measure = KZ_MEASURE_DISCRETE; b.eta = 1.0f;
            return mk3(1.0f);
        case KZ_BSDF_LAMBERTIAN:                                                             /* bsdf.cpp:241-257 */
            if (b.wi.z <= 0) return mk3(0.f);
            b.measure = KZ_MEASURE_SOLID_ANGLE;
            b.wo = square_to_cosine_hemisphere(sample2);
            b.eta = 1.0f;
            w = kz_tex_uv<FILT>(sc, m.base_color, b.uv, duv);
            break;
        case KZ_BSDF_GGX: {                                                                  /* bsdf.cpp:659-670 + ggx_brdf.h:175-203 (measure / eta keep their defaults) */
            if (b.wi.z <= 0) return mk3(0.f);
            const kz3 albedo = kz_tex_uv<FILT>(sc, m.base_color, b.uv, duv);
            const kz2 alpha = roughness_to_alpha(m.alpha, m.anisotropy);
            const kz3 H = sample_ggx_vndf(b.wi, alpha, sample2);
            b.wo = reflect3(b.wi, H);
            const float pdf = ggx_vndf(b.wi, H, alpha) / (4.0f * dot(b.wi, H));
            const kz3 color = ggx_smith_brdf(b.wi, b.wo, albedo, m.alpha, m.anisotropy);
            if (b.wo.z <= 0) return mk3(0.f);
            w = color * b.wo.z / pdf;
            break;
        }
        case KZ_BSDF_ROUGHCONDUCTOR: {                                                       /* bsdf.cpp:788-799 */
            if (b.wi.z <= 0) return mk3(0.f);
            const kz3 wh = square_to_beckmann(sample2, m.alpha);
            b.wo = normalized(reflect3(b.wi, wh));
            if (b.wo.z <= 0) return mk3(0.f);
            const float p = extra_pdf(m, b);
            *pdf_out = p;
            return extra_eval(sc, m, b) / p;
        }
        case KZ_BSDF_ROUGHPLASTIC: {                                                         /* bsdf.cpp:905-918 */
            if (b.wi.z <= 0) return mk3(0.f);
            const float ks = 1 - kd_max(m);
            if (sample1 < ks) {
                const kz3 wh = square_to_beckmann(sample2, m.alpha);
                b.wo = normalized((2.f * dot(wh, b.wi) * wh) - b.wi);
            } else b.wo = square_to_cosine_hemisphere(sample2);
            if (b.wo.z <= 0) return mk3(0.f);
            const float p = extra_pdf(m, b);
            *pdf_out = p;
            return extra_eval(sc, m, b) / p;
        }
        case KZ_BSDF_ROUGHDIELECTRIC: {                                                      /* bsdf.cpp:1050-1096 */
            const float m_eta = m.int_ior / m.ext_ior, m_invEta = m.ext_ior / m.int_ior;
            const float alpha = m.alpha * (1.2f - 0.2f * sqrtf(fabsf(b.wi.z)));
            const kz3 wm = square_to_beckmann(sample2, alpha);
            const float pdf = square_to_beckmann_pdf(wm, alpha);
            if (pdf == 0.f) return mk3(0.f);
            float cosThetaT;
            const float F = fresnel_dielectric(dot(b.wi, wm), m_eta, cosThetaT);
            if (!(sample1 > F)) {
                b.wo = reflect3(b.wi, wm);
                b.eta = 1.0f;
                if (b.wi.z * b.wo.z <= 0) return mk3(0.f);
            } else {
                if (cosThetaT == 0) return mk3(0.f);
                const float e = cosThetaT < 0 ? 1.f / m_eta : m_eta;                          /* RoughDielectric::refract, bsdf.cpp:1135-1139 */
                b.wo = wm * (dot(b.wi, wm) * e + cosThetaT) - b.wi * e;
                b.eta = cosThetaT < 0.f ? m_eta : m_invEta;
                if (b.wi.z * b.wo.z >= 0) return mk3(0.f);
            }
            const float D = beckmann_d(wm, alpha);
            const float G = beckmann_g1(b.wo, wm, alpha) * beckmann_g1(b.wi, wm, alpha);
            w = mk3(fabsf(D * G * dot(b.wi, wm) / (pdf * b.wi.z)));
            break;
        }
        default: return mk3(0.f);
    }
    *pdf_out = extra_pdf(m, b);
    return w;
}
KZ_HD_NOINLINE kz3 extra_sample(const KzScene &sc, const kz_bsdf_desc &m, KzBRec &b, float sample1, kz2 sample2, float *pdf_out) {
    return extra_sample_body<false>(sc, m, b, sample1, sample2, pdf_out, KzUvDiff{0.f, 0.f, 0.f, 0.f});
}
KZ_HD_NOINLINE kz3 extra_sample(const KzScene &sc, const kz_bsdf_desc &m, KzBRec &b, float sample1, kz2 sample2, float *pdf_out, KzUvDiff duv) {
    return extra_sample_body<true>(sc, m, b, sample1, sample2, pdf_out, duv);
}

/* One shading vertex: the hit mesh's BSDF with its (single) optional normal-map wrapper resolved.
 * Supported nesting (everything kazen's scenes use): diffuse | kiss | normalmap(diffuse|kiss). */
template <bool FILT> struct KzBsdfFoot {};
template <> struct KzBsdfFoot<true> { KzUvDiff duv; };     /* the vertex's footprint, which filters every uv-mode image lookup of its textures */
template <bool FILT = false>
struct KzBsdfCtx : KzBsdfFoot<FILT> {                       /* FILT = false: no footprint (an empty base takes no room) */
    const KzScene *sc;
    const kz_bsdf_desc *outer;     /* mesh BSDF */
    const kz_bsdf_desc *leaf;      /* nested (== outer when not a normal map) */
    KzKissParams kp;               /* leaf kiss parameters at uv */
    int leaf_type;                 /* leaf->type; a literal in the class-specialised shade kernels */
    bool is_nmap;
    kz3 nm_n;                      /* 2*rgb-1, un-normalised */
    KzFrame pert;                  /* perturbed frame (bsdf.cpp:366-374) */
};
/* CLS: material class the caller's queue was sorted into (KZ_CLASS_*), or -1 when unknown; a known
 * class turns the BSDF dispatch below into compile-time constants.  FILT: textures are filtered by the footprint `duv`. */
template <int CLS = -1, bool FILT = false>
KZ_HD KzBsdfCtx<FILT> bsdf_ctx(const KzScene &sc, const KzIts &its, const KzUvDiff &duv = KzUvDiff{0.f, 0.f, 0.f, 0.f}) {
    KzBsdfCtx<FILT> c;
    c.sc = &sc;
    if constexpr (FILT) c.duv = duv;
    c.outer = sc.bsdfs + sc.meshes[its.mesh].bsdf;
    c.is_nmap = CLS == KZ_CLASS_NORMALMAP ? true : (CLS >= 0 ? false : c.outer->type == KZ_BSDF_NORMALMAP);
    c.leaf = c.is_nmap ? sc.bsdfs + c.outer->nested : c.outer;
    c.leaf_type = CLS == KZ_CLASS_DIFFUSE ? KZ_BSDF_DIFFUSE : (CLS == KZ_CLASS_KISS ? KZ_BSDF_KISS : c.leaf->type);
    if (c.leaf_type == KZ_BSDF_KISS) c.kp = kiss_params<FILT>(sc, *c.leaf, its.uv, duv);
    else { c.kp.base = mk3(0.f); c.kp.metallic = 0.f; c.kp.roughness_raw = 0.f; }
    if (c.is_nmap) {
        kz3 rgb = kz_tex_uv<FILT>(sc, c.outer->normal_map, its.uv, duv);
        c.nm_n = mk3(2 * rgb.x - 1, 2 * rgb.y - 1, 2 * rgb.z - 1);
        kz3 n = normalized(c.nm_n);
        c.pert.n = normalized(to_world(its.sh, n));
        c.pert.s = normalized(its.dpdu - c.pert.n * dot(c.pert.n, its.dpdu));
        c.pert.t = normalized(cross(c.pert.n, c.pert.s));
    } else {
        c.nm_n = mk3(0.f, 0.f, 1.f);
        c.pert = its.sh;
    }
    return c;
}
template <bool FILT>
KZ_HD kz3 leaf_eval(const KzBsdfCtx<FILT> &c, const KzBRec &b) {
    if (c.leaf_type == KZ_BSDF_KISS) return kiss_eval(*c.leaf, c.kp, b);
    if (c.leaf_type > KZ_BSDF_NORMALMAP) {
        if constexpr (FILT) return extra_eval(*c.sc, *c.leaf, b, c.duv);
        else return extra_eval(*c.sc, *c.leaf, b);
    }
    if (b.measure != KZ_MEASURE_SOLID_ANGLE || b.wi.z <= 0 || b.wo.z <= 0) return mk3(0.0f);   /* bsdf.cpp:27-36 */
    return mk3(c.leaf->albedo[0], c.leaf->albedo[1], c.leaf->albedo[2]) * KZ_INV_PI * b.wo.z;
}
template <bool FILT>
KZ_HD float leaf_pdf(const KzBsdfCtx<FILT> &c, const KzBRec &b) {
    if (c.leaf_type == KZ_BSDF_KISS) return kiss_pdf(*c.leaf, c.kp, b);
    if (c.leaf_type > KZ_BSDF_NORMALMAP) return extra_pdf(*c.leaf, b);
    if (b.measure != KZ_MEASURE_SOLID_ANGLE || b.wi.z <= 0 || b.wo.z <= 0) return 0.0f;        /* bsdf.cpp:39-55 */
    return KZ_INV_PI * b.wo.z;
}
template <bool FILT>
KZ_HD kz3 leaf_sample(const KzBsdfCtx<FILT> &c, KzBRec &b, float s1, kz2 s2, float *pdf_out) {
    if (c.leaf_type == KZ_BSDF_KISS) return kiss_sample(*c.leaf, c.kp, b, s1, s2, pdf_out);
    if (c.leaf_type > KZ_BSDF_NORMALMAP) {
        if constexpr (FILT) return extra_sample(*c.sc, *c.leaf, b, s1, s2, pdf_out, c.duv);
        else return extra_sample(*c.sc, *c.leaf, b, s1, s2, pdf_out);
    }
    *pdf_out = 0.f;                                                                            /* bsdf.cpp:58-75 */
    if (b.wi.z <= 0) return mk3(0.0f);
    b.measure = KZ_MEASURE_SOLID_ANGLE;
    b.wo = square_to_cosine_hemisphere(s2);
    b.eta = 1.0f;
    *pdf_out = leaf_pdf(c, b);
    return mk3(c.leaf->albedo[0], c.leaf->albedo[1], c.leaf->albedo[2]);
}

/* eval + pdf of the mesh BSDF for (wi, wo) given in the ORIGINAL shading frame (NEE, integrator.cpp:283-290) */
template <bool FILT>
KZ_HD void bsdf_eval_pdf(const KzBsdfCtx<FILT> &c, const KzIts &its, kz3 wi, kz3 wo, kz3 *f, float *pdf) {
    KzBRec b; b.wi = wi; b.wo = wo; b.uv = its.uv; b.acc_rough = its.acc_rough; b.eta = 1.f; b.measure = KZ_MEASURE_SOLID_ANGLE;
    if (!c.is_nmap) { *f = leaf_eval(c, b); *pdf = leaf_pdf(c, b); return; }
    /* bsdf.cpp:290-336 */
    if (wi.z > 0 && wo.z > 0 && dot(c.nm_n, wi) <= 0) { *f = leaf_eval(c, b); *pdf = leaf_pdf(c, b); return; }
    KzBRec pq = b;
    pq.wi = to_local(c.pert, to_world(its.sh, wi));
    pq.wo = to_local(c.pert, to_world(its.sh, wo));
    pq.acc_rough = 0.f;                                  /* nested query carries a default `its` */
    if (wo.z * pq.wo.z <= 0) { *f = mk3(0.f); *pdf = 0.f; return; }
    *f = leaf_eval(c, pq); *pdf = leaf_pdf(c, pq);
}

/* sample() of the mesh BSDF + the integrator's follow-up pdf(bRec) query (integrator.cpp:307-314).
 * wo is returned in the ORIGINAL shading frame. */
template <bool FILT>
KZ_HD kz3 bsdf_sample(const KzBsdfCtx<FILT> &c, const KzIts &its, kz3 wi, float s1, kz2 s2, kz3 *wo, float *pdf, int *measure, float *eta) {
    KzBRec b; b.wi = wi; b.wo = mk3(0.f); b.uv = its.uv; b.acc_rough = its.acc_rough; b.eta = 1.f; b.measure = KZ_MEASURE_UNKNOWN;
    if (!c.is_nmap || (wi.z > 0 && dot(c.nm_n, wi) <= 0)) {
        float p;
        kz3 w = leaf_sample(c, b, s1, s2, &p);
        *wo = b.wo; *measure = b.measure; *eta = b.eta;
        /* integrator's pdf(bRec): for a normal map this re-enters NormalMap::pdf with the sampled wo */
        if (c.is_nmap && !iszero(w)) { kz3 f; bsdf_eval_pdf(c, its, wi, b.wo, &f, &p); }
        *pdf = p;
        return w;
    }
    /* bsdf.cpp:343-362 */
    KzBRec pq = b;
    pq.wi = to_local(c.pert, to_world(its.sh, wi));
    pq.acc_rough = 0.f;
    float p;
    kz3 result = leaf_sample(c, pq, s1, s2, &p);
    *measure = KZ_MEASURE_UNKNOWN;          /* bRec.measure is never written back on this path */
    *pdf = 0.f; *eta = 1.f;
    if (!iszero(result)) {
        kz3 w = to_local(its.sh, to_world(c.pert, pq.wo));
        *wo = w; *eta = pq.eta;
        if (w.z * pq.wo.z <= 0) return mk3(0.f);
        /* integrator's pdf(bRec) with measure == unknown: kiss ignores the measure, diffuse returns 0 */
        KzBRec q = b; q.wo = w;
        if (wi.z > 0 && w.z > 0 && dot(c.nm_n, wi) <= 0) *pdf = leaf_pdf(c, q);
        else {
            KzBRec pq2 = q;
            pq2.wi = pq.wi; pq2.wo = to_local(c.pert, to_world(its.sh, w)); pq2.acc_rough = 0.f;
            *pdf = (w.z * pq2.wo.z <= 0) ? 0.f : leaf_pdf(c, pq2);
        }
    }
    return result;
}
template <bool FILT>
KZ_HD float bsdf_regularize(const KzBsdfCtx<FILT> &c) {   /* bsdf.h:125, bsdf.cpp:412,1397-1399 */
    return c.leaf_type == KZ_BSDF_KISS ? c.kp.roughness_raw : 0.f;
}

/* ---- lights -------------------------------------------------------------------------------- */
KZ_HD KzVertex kz_vertex(const KzScene &sc, const KzMeshRec &m, uint32_t i) { return sc.vertices[(size_t)m.vertex_offset + i]; }
KZ_HD kz3 kz_vpos(const KzVertex &v) { return mk3(v.px, v.py, v.pz); }
KZ_HD kz3 kz_vnrm(const KzVertex &v) { return mk3(v.nx, v.ny, v.nz); }
KZ_HD kz2 kz_vuv(const KzVertex &v) { return mk2(v.u, v.v); }

/* dpdf.h:99-104: std::lower_bound over cdf[0..n], then index = clamp(pos-1, 0, n-1) */
KZ_HD uint32_t cdf_sample(const float *cdf, uint32_t n, float v) {
    uint32_t lo = 0, hi = n + 1;                 /* first element >= v in [0, n+1) */
    while (lo < hi) {
        uint32_t mid = (lo + hi) >> 1;
        if (cdf[mid] < v) lo = mid + 1; else hi = mid;
    }
    int32_t idx = (int32_t)lo - 1;
    if (idx < 0) idx = 0;
    return (uint32_t)idx < n - 1 ? (uint32_t)idx : n - 1;
}
/* light.cpp:16-19,36-51 */
KZ_HD float light_pdf(float inv_area, kz3 ref, kz3 p, kz3 n, kz3 wi) {
    float cosTheta = dot(n, -wi);
    if (cosTheta > 0.f) return inv_area * sqnorm(p - ref) / cosTheta;
    return 0.f;
}

/* ---- post-intersection (accel.cpp:113-236) ---------------------------------------------- */
KZ_HD void fill_intersection(const KzScene &sc, const KzHit &h, KzIts &its, kz3 prev_dpdu) {
    its.mesh = (int32_t)h.geom;
    const KzMeshRec m = sc.meshes[h.geom];
    const KzU4 F = sc.indices[(size_t)m.index_offset + h.prim];
    const KzVertex v0 = kz_vertex(sc, m, F.x), v1 = kz_vertex(sc, m, F.y), v2 = kz_vertex(sc, m, F.z);
    const float b0 = 1 - (h.u + h.v), b1 = h.u, b2 = h.v;
    const bool hasN = (m.flags & KZ_MESH_HAS_NORMALS) != 0, hasUV = (m.flags & KZ_MESH_HAS_UVS) != 0;
    const kz3 p0 = kz_vpos(v0), p1 = kz_vpos(v1), p2 = kz_vpos(v2);
    kz3 n0 = mk3(0.f), n1 = mk3(0.f), n2 = mk3(0.f);
    if (hasN) { n0 = kz_vnrm(v0); n1 = kz_vnrm(v1); n2 = kz_vnrm(v2); }
    const kz3 orignP = b0 * p0 + b1 * p1 + b2 * p2;
    kz3 tmpu = orignP - p0, tmpv = orignP - p1, tmpw = orignP - p2;
    const float dotu = fminf(0.f, dot(tmpu, n0)), dotv = fminf(0.f, dot(tmpv, n1)), dotw = fminf(0.f, dot(tmpw, n2));
    tmpu -= dotu * n0; tmpv -= dotv * n1; tmpw -= dotw * n2;
    its.p = orignP + b0 * tmpu + b1 * tmpv + b2 * tmpw;
    const kz3 dp0 = p1 - p0, dp1 = p2 - p0;
    const kz3 gcross = cross(dp0, dp1);
    its.geo_n = normalized(gcross);
    its.uv = mk2(h.u, h.v);
    its.dpdu = prev_dpdu;
    kz2 uv0 = mk2(0, 0), uv1 = mk2(0, 0), uv2 = mk2(0, 0);
    if (hasUV) {
        uv0 = kz_vuv(v0); uv1 = kz_vuv(v1); uv2 = kz_vuv(v2);
        its.uv = mk2(b0 * uv0.x + b1 * uv1.x + b2 * uv2.x, b0 * uv0.y + b1 * uv1.y + b2 * uv2.y);
    }
    if (hasN && hasUV) {
        const kz2 duv0 = mk2(uv1.x - uv0.x, uv1.y - uv0.y), duv1 = mk2(uv2.x - uv0.x, uv2.y - uv0.y);
        const kz3 shNormal = b0 * n0 + b1 * n1 + b2 * n2;
        const float length = norm(gcross);
        if (length > 0.f) {
            const float determinant = duv0.x * duv1.y - duv0.y * duv1.x;
            if (determinant > 0.f) {
                const float invDet = 1.0f / determinant;
                its.dpdu = (duv1.y * dp0 - duv0.y * dp1) * invDet;
                its.sh.n = normalized(shNormal);
                its.sh.s = normalized(its.dpdu - shNormal * dot(shNormal, its.dpdu));
                its.sh.t = normalized(cross(its.sh.n, its.sh.s));
            } else {
                its.sh = frame_from_normal(normalized(shNormal));
                its.dpdu = its.sh.s;
            }
        } else {
            its.sh = frame_from_normal(normalized(shNormal));
        }
    } else if (hasN) {
        its.sh = frame_from_normal(normalized(b0 * n0 + b1 * n1 + b2 * n2));
    } else {
        its.sh = frame_from_normal(its.geo_n);
    }
}

#endif
