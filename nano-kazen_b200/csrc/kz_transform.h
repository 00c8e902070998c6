/* kz_transform.h -- the per-vertex body of kzgpu_mesh_transform: a rest-pose position and normal placed by a row-major 4x4 matrix and
 * its inverse, rounded as the C++ host's OBJ loader rounds them when it applies `toWorld` (so a mesh transformed on the GPU equals the
 * same file loaded with that transform, bit for bit):
 *
 *   kz_transform_point    Transform::point (host/src/core.cpp:53-60): each row ((M0 x + M1 y) + M2 z) + M3, then x, y, z divided by w
 *   kz_transform_normal   Transform::normal (core.cpp:65-68): the transpose of the inverse's upper 3x3 times n, then the loader's
 *                         normalisation (plugins.cpp:533-535): z = x^2 + (y^2 + z^2), n / sqrt(z) when z > 0, else n as it is
 *
 * Every operation is one kz_mul / kz_add / kz_div / kz_sqrt, so nvcc cannot contract a product and a sum into one FFMA.  The KZ_HD
 * functions are compiled by g++ for tests/hostemu (transform_emu.cpp) and by the host pass of kz_api.cu (emitter tables) as well;
 * k_transform_vertices (kz_ingest.cuh) wraps them in a kernel. */
#ifndef KZ_TRANSFORM_H
#define KZ_TRANSFORM_H
#include "kz_common.h"

/* a matrix and the inverse it is paired with, row-major, passed to the kernel by value */
struct KzXform { float m[16], inv[16]; };

KZ_HD void kz_transform_point(const float *M, const float *p, float *out) {
    float r[4];
    for (int i = 0; i < 4; ++i)
        r[i] = kz_add(kz_add(kz_add(kz_mul(M[4 * i], p[0]), kz_mul(M[4 * i + 1], p[1])), kz_mul(M[4 * i + 2], p[2])), M[4 * i + 3]);
    out[0] = kz_div(r[0], r[3]); out[1] = kz_div(r[1], r[3]); out[2] = kz_div(r[2], r[3]);
}

KZ_HD void kz_transform_normal(const float *I, const float *n, float *out) {
    float r[3];
    for (int j = 0; j < 3; ++j) r[j] = kz_add(kz_add(kz_mul(I[j], n[0]), kz_mul(I[4 + j], n[1])), kz_mul(I[8 + j], n[2]));
    const float z = kz_add(kz_mul(r[0], r[0]), kz_add(kz_mul(r[1], r[1]), kz_mul(r[2], r[2])));
    if (z > 0.f) {
        const float l = kz_sqrt(z);
        r[0] = kz_div(r[0], l); r[1] = kz_div(r[1], l); r[2] = kz_div(r[2], l);
    }
    out[0] = r[0]; out[1] = r[1]; out[2] = r[2];
}

#endif
