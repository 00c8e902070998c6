/* kz_env.cuh -- the environment table of kz_env.h built on the GPU at kzgpu_scene_upload, and its sampling probe.  The per-item
 * bodies are kz_env.h's; the sums run sequentially in double (one thread per row, one for the marginal), so every device builds the
 * same bytes. */
#ifndef KZ_ENV_CUH
#define KZ_ENV_CUH
#include "kz_env.h"

__global__ void k_env_weights(KzScene sc, KzEnvChain ch, const double *row_sin, int w, int h, double *weight) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)w * h) return;
    weight[i] = kz_env_cell_weight(sc, ch, row_sin, w, h, (int)(i % (size_t)w), (int)(i / (size_t)w));
}
__global__ void k_env_rows(const double *weight, int w, int h, float *cdf, double *row_sum) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= h) return;
    row_sum[r] = kz_env_row(weight + (size_t)r * w, w, cdf + (size_t)r * (w + 1));
}
__global__ void k_env_marginal(const double *row_sum, int h, float *cdf, double *total) {
    if (blockIdx.x == 0 && threadIdx.x == 0) *total = kz_env_marginal(row_sum, h, cdf);
}
__global__ void k_env_probs(const double *weight, size_t n, const double *total, float *prob) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) prob[i] = kz_env_cell_prob(weight[i], *total);
}

/* kzgpu_env_sample_dump: direction, density, radiance per (row draw, column draw) */
__global__ void k_env_sample_dump(KzScene sc, KzEnvTable env, const float *u2, uint32_t n, float *out8) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const kz3 d = kz_env_sample(env, u2[2 * (size_t)i], u2[2 * (size_t)i + 1]);
    const kz3 le = kz_background(sc, d);
    float *o = out8 + 8 * (size_t)i;
    o[0] = d.x; o[1] = d.y; o[2] = d.z; o[3] = kz_env_pdf(env, d);
    o[4] = le.x; o[5] = le.y; o[6] = le.z; o[7] = 0.f;
}

#endif
