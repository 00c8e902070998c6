/* kz_env.h -- the environment as a light for path_mis (kz_integrator_desc::env_sampling): the background chain's kind, the per-item
 * bodies of its luminance table (built on the GPU by the kernels of kz_env.cuh, and on the host by tests/hostemu/env_emu.cpp), and
 * sampling / density over that table.
 *
 * Table (W x H cells over the lat-long square (s, t) of kz_tex_eval_tree's direction lookup; row r = t in [r/H, (r+1)/H)):
 *   weight(c, r) = max |luminance| of the 5 x 5 texels kz_image_bicubic can read for a point of the cell (wrapped in s and t as the
 *                  lookup wraps; the texels as stored: the direction lookup applies neither sRGB conversion nor scale), times sin(theta)
 *                  at the row centre.  A constant chain uses a 64 x 32 grid of weight sin(theta).  The weight is positive wherever the
 *                  lookup can return a non-zero value, so every direction the background lights has a positive density.
 *   row CDFs, the marginal over rows and the cell probabilities are summed sequentially in double and rounded to float once: the table
 *   is the same bytes on every device and on the host.
 * Density: pdf(w) = p_cell * W * H / (2 pi^2 cos(lambda)), lambda = elevation (the Jacobian of the lat-long map). */
#ifndef KZ_ENV_H
#define KZ_ENV_H
#include "kz_shade.h"

#define KZ_ENV_ZERO 0          /* the background evaluates to 0 in every direction (none, zero intensity, colorramp / blend, cut off) */
#define KZ_ENV_CONSTANT 1      /* it evaluates to one non-zero colour */
#define KZ_ENV_IMAGE 2         /* it ends in an image texture, looked up by direction */
#define KZ_ENV_CONST_W 64
#define KZ_ENV_CONST_H 32

/* The table as the sampling kernels read it.  Kept out of KzScene (a trailing parameter of k_shade instead): the scene is the
 * parameter of every kernel, and the flag-off kernels keep their code by keeping its layout. */
struct KzEnvTable {
    const float *cdf;          /* h rows of w + 1 floats: the CDF over the row's cells */
    const float *marginal;     /* h + 1 floats: the CDF over rows                      */
    const float *prob;         /* w * h floats: the probability of each cell           */
    int32_t w, h;
};

/* exactly rounded double arithmetic (never contracted), as kz_mul / kz_add are for float */
#if KZ_DEVICE_CODE
KZ_HD double kz_dmul(double a, double b) { return __dmul_rn(a, b); }
KZ_HD double kz_dadd(double a, double b) { return __dadd_rn(a, b); }
KZ_HD double kz_ddiv(double a, double b) { return __ddiv_rn(a, b); }
#else
KZ_HD double kz_dmul(double a, double b) { volatile double r = a * b; return r; }
KZ_HD double kz_dadd(double a, double b) { volatile double r = a + b; return r; }
KZ_HD double kz_ddiv(double a, double b) { volatile double r = a / b; return r; }
#endif

/* The background chain walked by the rules of kz_tex_eval_tree's direction mode: a background node forwards to child 0 and scales by
 * its intensity, a missing child or the KZ_TEX_MAX_DEPTH cut-off evaluates to 0, colorramp and blend evaluate to 0 by direction. */
struct KzEnvChain { int32_t kind, image; };
KZ_HD KzEnvChain kz_env_classify(const KzScene &sc) {
    KzEnvChain r; r.kind = KZ_ENV_ZERO; r.image = -1;
    if (sc.background < 0) return r;
    int node = sc.background;
    float scale = 1.f;
    for (int depth = 0;; ++depth) {
        const kz_texture_desc t = sc.textures[node];
        if (t.type == KZ_TEX_BACKGROUND) {
            if (t.child[0] < 0 || depth + 1 == KZ_TEX_MAX_DEPTH) return r;
            scale *= t.a;
            node = t.child[0];
            continue;
        }
        if (t.type == KZ_TEX_IMAGE && scale != 0.f) { r.kind = KZ_ENV_IMAGE; r.image = t.image; }
        if (t.type == KZ_TEX_CONSTANT && !iszero(kz_background(sc, mk3(0.f, 0.f, 1.f)))) r.kind = KZ_ENV_CONSTANT;
        return r;
    }
}
KZ_HD void kz_env_dims(const KzScene &sc, const KzEnvChain &ch, int &w, int &h) {
    if (ch.kind == KZ_ENV_IMAGE) { w = sc.images[ch.image].width; h = sc.images[ch.image].height; }
    else { w = KZ_ENV_CONST_W; h = KZ_ENV_CONST_H; }
}
/* sin(theta) at the centre of every row, in double (host libm: the same values wherever the table is built) */
inline void kz_env_row_sines(int h, double *out) {
    for (int r = 0; r < h; ++r) out[r] = sin(3.14159265358979323846 * ((double)r + 0.5) / (double)h);
}

/* ---- table: one cell, one row, the marginal, one cell probability ---------------------------------------------------------------- */
KZ_HD double kz_env_luminance_abs(const KzF4 &p) {      /* the float products are exact in double */
    const double l = kz_dadd(kz_dadd(kz_dmul((double)p.x, (double)0.212671f), kz_dmul((double)p.y, (double)0.715160f)), kz_dmul((double)p.z, (double)0.072169f));
    return l < 0.0 ? -l : l;
}
KZ_HD double kz_env_cell_weight(const KzScene &sc, const KzEnvChain &ch, const double *row_sin, int w, int h, int c, int r) {
    double m = 1.0;
    if (ch.kind == KZ_ENV_IMAGE) {
        const KzF4 *base = sc.texels + sc.images[ch.image].texel_offset;
        m = 0.0;
        for (int j = -2; j <= 2; ++j) {
            const int yy = kz_wrapi(r + j, h);
            for (int i = -2; i <= 2; ++i) {
                const double l = kz_env_luminance_abs(base[(size_t)yy * w + kz_wrapi(c + i, w)]);
                m = l > m ? l : m;
            }
        }
    }
    return kz_dmul(m, row_sin[r]);
}
/* row r of the weights (w doubles) -> its CDF (w + 1 floats, 0 .. 1; uniform for an empty row); returns the row's sum */
KZ_HD double kz_env_row(const double *weight, int w, float *cdf) {
    double sum = 0.0;
    for (int c = 0; c < w; ++c) sum = kz_dadd(sum, weight[c]);
    double acc = 0.0;
    cdf[0] = 0.f;
    for (int c = 0; c < w; ++c) {
        acc = kz_dadd(acc, weight[c]);
        cdf[c + 1] = sum > 0.0 ? (float)kz_ddiv(acc, sum) : (float)kz_ddiv((double)(c + 1), (double)w);
    }
    cdf[w] = 1.f;
    return sum;
}
/* the row sums (h doubles) -> the marginal CDF (h + 1 floats); returns the table total */
KZ_HD double kz_env_marginal(const double *row_sum, int h, float *cdf) {
    double total = 0.0;
    for (int r = 0; r < h; ++r) total = kz_dadd(total, row_sum[r]);
    double acc = 0.0;
    cdf[0] = 0.f;
    for (int r = 0; r < h; ++r) {
        acc = kz_dadd(acc, row_sum[r]);
        cdf[r + 1] = total > 0.0 ? (float)kz_ddiv(acc, total) : (float)kz_ddiv((double)(r + 1), (double)h);
    }
    cdf[h] = 1.f;
    return total;
}
KZ_HD float kz_env_cell_prob(double weight, double total) { return total > 0.0 ? (float)kz_ddiv(weight, total) : 0.f; }

/* ---- sampling and density ------------------------------------------------------------------------------------------------------ */
/* (s, t) -> direction: the inverse of s = atan2(-d.x, d.z) / 2pi + 0.5, t = 0.5 - atan2(d.y, hypot(d.z, -d.x)) / pi */
KZ_HD kz3 kz_env_dir(float s, float t) {
    const float phi = (s - 0.5f) * (2.0f * KZ_PI), lambda = (0.5f - t) * KZ_PI;
    const float cl = cosf(lambda);
    return mk3(-cl * sinf(phi), sinf(lambda), cl * cosf(phi));
}
/* solid-angle density of kz_env_sample at direction d (the miss branch and the light sample both use this) */
KZ_HD float kz_env_pdf(const KzEnvTable &env, kz3 d) {
    float s = atan2f(-d.x, d.z) / (2.0f * KZ_PI) + 0.5f;
    float t = 0.5f - atan2f(d.y, hypotf(d.z, -d.x)) / KZ_PI;
    if (isnan(s)) s = 0.0f;
    if (isnan(t)) t = 0.0f;
    const float hz = hypotf(d.z, -d.x), len = sqrtf(hz * hz + d.y * d.y);
    const float cl = hz / len;                                 /* cos(elevation) */
    if (!(cl > 0.f)) return 0.f;
    const int w = env.w, h = env.h;
    int c = (int)(s * (float)w), r = (int)(t * (float)h);
    c = c < 0 ? 0 : (c > w - 1 ? w - 1 : c);
    r = r < 0 ? 0 : (r > h - 1 ? h - 1 : r);
    return env.prob[(size_t)r * w + c] * ((float)w * (float)h) / ((2.0f * KZ_PI * KZ_PI) * cl);
}
/* Distribution2D::SampleContinuous (pbrt): u_row picks the row through the marginal, u_col the column through the row's CDF, and the
 * remainders place the point inside the cell */
KZ_HD kz3 kz_env_sample(const KzEnvTable &env, float u_row, float u_col) {
    const uint32_t w = (uint32_t)env.w, h = (uint32_t)env.h;
    const uint32_t r = cdf_sample(env.marginal, h, u_row);
    const float m0 = env.marginal[r], m1 = env.marginal[r + 1];
    float dv = u_row - m0;
    if (m1 - m0 > 0.f) dv /= (m1 - m0);
    const float *row = env.cdf + (size_t)r * (w + 1);
    const uint32_t c = cdf_sample(row, w, u_col);
    const float c0 = row[c], c1 = row[c + 1];
    float du = u_col - c0;
    if (c1 - c0 > 0.f) du /= (c1 - c0);
    return kz_env_dir(((float)c + du) / (float)w, ((float)r + dv) / (float)h);
}

#endif
