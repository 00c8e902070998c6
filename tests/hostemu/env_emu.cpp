/* tests/hostemu/env_emu.cpp -- DEVELOPMENT/TEST HARNESS, NOT A PRODUCT PATH.
 *
 * emu.cpp (the device routines compiled for the host) plus the environment table of kz_env.h, built with the same per-item bodies the
 * kernels of kz_env.cuh run (cell weights, one row at a time, the marginal, the cell probabilities), and its sampling and density.
 * Built as its own library (env_emu.py) so that the CPU suite can check the table against a numpy restatement and the sampler
 * against the table.
 */
#include "emu.cpp"
#include "../../nano-kazen_b200/csrc/kz_env.h"

struct kzenv {
    kzemu *e = nullptr;
    KzEnvChain chain{KZ_ENV_ZERO, -1};
    KzEnvTable env{nullptr, nullptr, nullptr, 0, 0};
    std::vector<float> cdf, marginal, prob;
    double total = 0.0;
};

extern "C" {

/* The emulation of `d` with its environment table (built whatever the integrator and env_sampling say, for any chain but ZERO). */
int kzenv_create(const kz_scene_desc *d, kzenv **out) {
    kzenv *v = new kzenv();
    int rc = kzemu_create(d, &v->e);
    if (rc) { delete v; return rc; }
    KzScene &sc = v->e->hs.sc;
    v->chain = kz_env_classify(sc);
    if (v->chain.kind != KZ_ENV_ZERO) {
        int w, h;
        kz_env_dims(sc, v->chain, w, h);
        std::vector<double> sines((size_t)h), weight((size_t)w * h), row_sum((size_t)h);
        kz_env_row_sines(h, sines.data());
        for (int r = 0; r < h; ++r)
            for (int c = 0; c < w; ++c) weight[(size_t)r * w + c] = kz_env_cell_weight(sc, v->chain, sines.data(), w, h, c, r);
        v->cdf.resize((size_t)h * (w + 1)); v->marginal.resize((size_t)h + 1); v->prob.resize((size_t)w * h);
        for (int r = 0; r < h; ++r) row_sum[(size_t)r] = kz_env_row(weight.data() + (size_t)r * w, w, v->cdf.data() + (size_t)r * (w + 1));
        v->total = kz_env_marginal(row_sum.data(), h, v->marginal.data());
        for (size_t i = 0; i < weight.size(); ++i) v->prob[i] = kz_env_cell_prob(weight[i], v->total);
        v->env = KzEnvTable{v->cdf.data(), v->marginal.data(), v->prob.data(), w, h};
    }
    *out = v;
    return KZ_OK;
}
void kzenv_destroy(kzenv *v) { if (v) { kzemu_destroy(v->e); delete v; } }

/* kind (KZ_ENV_*), table width and height, whether it counts (total > 0), and the total */
int kzenv_info(kzenv *v, int *kind, int *w, int *h, int *counted, double *total) {
    *kind = v->chain.kind; *w = v->env.w; *h = v->env.h; *counted = v->total > 0.0; *total = v->total;
    return KZ_OK;
}
/* the table: h * (w + 1) row CDF floats, h + 1 marginal floats, w * h cell probabilities */
int kzenv_table(kzenv *v, float *cdf, float *marginal, float *prob) {
    memcpy(cdf, v->cdf.data(), v->cdf.size() * 4); memcpy(marginal, v->marginal.data(), v->marginal.size() * 4); memcpy(prob, v->prob.data(), v->prob.size() * 4);
    return KZ_OK;
}
/* per direction (3 floats): kz_background (3 floats) and, with a table, kz_env_pdf */
int kzenv_eval(kzenv *v, const float *dirs, size_t n, float *rgb, float *pdf) {
    const KzScene &sc = v->e->hs.sc;
    pfor(n, [&](size_t b, size_t en) {
        for (size_t i = b; i < en; ++i) {
            const kz3 d = mk3(dirs[3 * i], dirs[3 * i + 1], dirs[3 * i + 2]);
            const kz3 c = kz_background(sc, d);
            rgb[3 * i] = c.x; rgb[3 * i + 1] = c.y; rgb[3 * i + 2] = c.z;
            if (pdf) pdf[i] = v->env.w > 0 ? kz_env_pdf(v->env, d) : 0.f;
        }
    });
    return KZ_OK;
}
/* kzgpu_env_sample_dump's layout: direction[3], density, radiance[3], 0 per (row draw, column draw) */
int kzenv_sample(kzenv *v, const float *u2, size_t n, float *out8) {
    const KzScene &sc = v->e->hs.sc;
    if (v->env.w == 0) return KZ_ERR_STATE;
    pfor(n, [&](size_t b, size_t en) {
        for (size_t i = b; i < en; ++i) {
            const kz3 d = kz_env_sample(v->env, u2[2 * i], u2[2 * i + 1]);
            const kz3 le = kz_background(sc, d);
            float *o = out8 + 8 * i;
            o[0] = d.x; o[1] = d.y; o[2] = d.z; o[3] = kz_env_pdf(v->env, d); o[4] = le.x; o[5] = le.y; o[6] = le.z; o[7] = 0.f;
        }
    });
    return KZ_OK;
}

}  // extern "C"
