/* kz_texlod.h -- texture footprint of a shading vertex for filtered lookups (kz_integrator_desc::texture_filtering).
 *
 * The path slots have no room for ray differentials (kz_path.h: blocks A, B and C are whole sectors), so the footprint is pbrt-v4's
 * stateless camera estimate (CameraBase::Approximate_dp_dxy + SurfaceInteraction::ComputeDifferentials): at any point the camera sees,
 * the pixel-step offsets on the tangent plane of the rays that leave the camera at the smallest angular step of the film (found once
 * on the host, kz_tex_lod), scaled by max(1/8, 1/sqrt(spp)).  It ignores how the path got there: a vertex after a bounce gets the
 * footprint the camera would see at that point.  That is pbrt-v4's known approximation; it errs towards sharp lookups (a footprint
 * seen through a curved mirror or after a diffuse bounce is wider than this). */
#ifndef KZ_TEXLOD_H
#define KZ_TEXLOD_H
#include "kz_shade.h"
#include <algorithm>
#include <cmath>

/* What the filtered shade kernels need besides the scene: rows 0-2 of camera_from_world (the inverse of camera_to_world, inverted in
 * double and rounded once), pbrt's minimum direction differentials in the frame of the central ray, and sppScale. */
struct KzTexLod {
    float camera_from_world[12];
    float ddx[3], ddy[3];
    float spp_scale;
};

/* ---- host: at kzgpu_scene_upload and kzgpu_camera_update ------------------------------------------------------------------- */
/* pbrt-v4's CoordinateSystem (Duff et al.): the frame Frame::FromZ builds around a unit vector */
inline void kz_lod_frame(const double z[3], double x[3], double y[3]) {
    const double sign = std::copysign(1.0, z[2]);
    const double a = -1.0 / (sign + z[2]);
    const double b = z[0] * z[1] * a;
    x[0] = 1.0 + sign * (z[0] * z[0]) * a; x[1] = sign * b; x[2] = -sign * z[0];
    y[0] = b; y[1] = sign + (z[1] * z[1]) * a; y[2] = -z[1];
}
/* camera-space direction of the pinhole ray through film point (fx, fy) (kz_camera_ray without the aperture: for a thin lens the ray
 * through the lens centre has this direction too), normalised */
inline void kz_lod_film_dir(const kz_camera_desc &c, double fx, double fy, double d[3]) {
    const double x = fx / (double)c.width, y = fy / (double)c.height;
    const float *M = c.sample_to_camera;
    double r[4];
    for (int i = 0; i < 4; ++i) r[i] = (double)M[4 * i] * x + (double)M[4 * i + 1] * y + (double)M[4 * i + 3];
    for (int i = 0; i < 3; ++i) d[i] = r[i] / r[3];
    const double n = std::sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
    for (int i = 0; i < 3; ++i) d[i] /= n;
}
/* CameraBase::FindMinimumDifferentials: 512 film points on the diagonal; at each, the rays through the point and the point + (1, 0) /
 * + (0, 1) expressed in the central ray's frame; the shortest local(d_x) - (0, 0, 1) and local(d_y) - (0, 0, 1) are kept.  The
 * position differentials of both camera types are 0 (the lens centre's rays share their origin). */
inline KzTexLod kz_tex_lod(const kz_camera_desc &c, uint32_t sample_count) {
    KzTexLod lod;
    double inv[16], m[16];
    for (int i = 0; i < 16; ++i) m[i] = c.camera_to_world[i];
    /* 4x4 inverse by cofactors, in double */
    inv[0] = m[5] * m[10] * m[15] - m[5] * m[11] * m[14] - m[9] * m[6] * m[15] + m[9] * m[7] * m[14] + m[13] * m[6] * m[11] - m[13] * m[7] * m[10];
    inv[4] = -m[4] * m[10] * m[15] + m[4] * m[11] * m[14] + m[8] * m[6] * m[15] - m[8] * m[7] * m[14] - m[12] * m[6] * m[11] + m[12] * m[7] * m[10];
    inv[8] = m[4] * m[9] * m[15] - m[4] * m[11] * m[13] - m[8] * m[5] * m[15] + m[8] * m[7] * m[13] + m[12] * m[5] * m[11] - m[12] * m[7] * m[9];
    inv[12] = -m[4] * m[9] * m[14] + m[4] * m[10] * m[13] + m[8] * m[5] * m[14] - m[8] * m[6] * m[13] - m[12] * m[5] * m[10] + m[12] * m[6] * m[9];
    inv[1] = -m[1] * m[10] * m[15] + m[1] * m[11] * m[14] + m[9] * m[2] * m[15] - m[9] * m[3] * m[14] - m[13] * m[2] * m[11] + m[13] * m[3] * m[10];
    inv[5] = m[0] * m[10] * m[15] - m[0] * m[11] * m[14] - m[8] * m[2] * m[15] + m[8] * m[3] * m[14] + m[12] * m[2] * m[11] - m[12] * m[3] * m[10];
    inv[9] = -m[0] * m[9] * m[15] + m[0] * m[11] * m[13] + m[8] * m[1] * m[15] - m[8] * m[3] * m[13] - m[12] * m[1] * m[11] + m[12] * m[3] * m[9];
    inv[13] = m[0] * m[9] * m[14] - m[0] * m[10] * m[13] - m[8] * m[1] * m[14] + m[8] * m[2] * m[13] + m[12] * m[1] * m[10] - m[12] * m[2] * m[9];
    inv[2] = m[1] * m[6] * m[15] - m[1] * m[7] * m[14] - m[5] * m[2] * m[15] + m[5] * m[3] * m[14] + m[13] * m[2] * m[7] - m[13] * m[3] * m[6];
    inv[6] = -m[0] * m[6] * m[15] + m[0] * m[7] * m[14] + m[4] * m[2] * m[15] - m[4] * m[3] * m[14] - m[12] * m[2] * m[7] + m[12] * m[3] * m[6];
    inv[10] = m[0] * m[5] * m[15] - m[0] * m[7] * m[13] - m[4] * m[1] * m[15] + m[4] * m[3] * m[13] + m[12] * m[1] * m[7] - m[12] * m[3] * m[5];
    inv[14] = -m[0] * m[5] * m[14] + m[0] * m[6] * m[13] + m[4] * m[1] * m[14] - m[4] * m[2] * m[13] - m[12] * m[1] * m[6] + m[12] * m[2] * m[5];
    inv[3] = -m[1] * m[6] * m[11] + m[1] * m[7] * m[10] + m[5] * m[2] * m[11] - m[5] * m[3] * m[10] - m[9] * m[2] * m[7] + m[9] * m[3] * m[6];
    inv[7] = m[0] * m[6] * m[11] - m[0] * m[7] * m[10] - m[4] * m[2] * m[11] + m[4] * m[3] * m[10] + m[8] * m[2] * m[7] - m[8] * m[3] * m[6];
    inv[11] = -m[0] * m[5] * m[11] + m[0] * m[7] * m[9] + m[4] * m[1] * m[11] - m[4] * m[3] * m[9] - m[8] * m[1] * m[7] + m[8] * m[3] * m[5];
    inv[15] = m[0] * m[5] * m[10] - m[0] * m[6] * m[9] - m[4] * m[1] * m[10] + m[4] * m[2] * m[9] + m[8] * m[1] * m[6] - m[8] * m[2] * m[5];
    const double det = m[0] * inv[0] + m[1] * inv[4] + m[2] * inv[8] + m[3] * inv[12];
    for (int i = 0; i < 12; ++i) lod.camera_from_world[i] = (float)(inv[i] / det);
    double best_x = HUGE_VAL, best_y = HUGE_VAL, dx[3] = {0, 0, 0}, dy[3] = {0, 0, 0};
    const int n = 512;
    for (int i = 0; i < n; ++i) {
        const double fx = (double)i / (n - 1) * c.width, fy = (double)i / (n - 1) * c.height;
        double d[3], rx[3], ry[3], fxv[3], fyv[3];
        kz_lod_film_dir(c, fx, fy, d);
        kz_lod_film_dir(c, fx + 1.0, fy, rx);
        kz_lod_film_dir(c, fx, fy + 1.0, ry);
        kz_lod_frame(d, fxv, fyv);
        for (int k = 0; k < 2; ++k) {
            const double *r = k == 0 ? rx : ry;
            double l[3] = {r[0] * fxv[0] + r[1] * fxv[1] + r[2] * fxv[2], r[0] * fyv[0] + r[1] * fyv[1] + r[2] * fyv[2], r[0] * d[0] + r[1] * d[1] + r[2] * d[2]};
            const double ln = std::sqrt(l[0] * l[0] + l[1] * l[1] + l[2] * l[2]);
            const double v[3] = {l[0] / ln, l[1] / ln, l[2] / ln - 1.0};
            const double len = std::sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
            double &best = k == 0 ? best_x : best_y;
            double *dst = k == 0 ? dx : dy;
            if (len < best) { best = len; dst[0] = v[0]; dst[1] = v[1]; dst[2] = v[2]; }
        }
    }
    for (int k = 0; k < 3; ++k) { lod.ddx[k] = (float)dx[k]; lod.ddy[k] = (float)dy[k]; }
    lod.spp_scale = (float)std::max(0.125, 1.0 / std::sqrt((double)sample_count));
    return lod;
}

/* ---- device: once per shaded vertex ---------------------------------------------------------------------------------------- */
KZ_HD float kz_lod_clamp(float v) { return isfinite(v) ? clampf(v, -1e8f, 1e8f) : 0.f; }
/* The uv derivatives per pixel step at point p (geometric normal n) of the triangle (p0, p1, p2) with texture coordinates (uv0, uv1,
 * uv2).  c2w: the camera's camera_to_world (row-major 4x4).  pbrt-v4's Approximate_dp_dxy gives dp/dx and dp/dy on the tangent plane;
 * they map to uv through the triangle's own barycentric Jacobian: the 2x2 Gram system of e1 = p1 - p0, e2 = p2 - p0 gives the
 * barycentric steps, and uv follows them linearly.  A singular system or a non-finite step gives 0; the rest is clamped to +-1e8. */
KZ_HD KzUvDiff kz_uv_footprint(const KzTexLod &lod, const float *c2w, kz3 p, kz3 n, kz3 p0, kz3 p1, kz3 p2, kz2 uv0, kz2 uv1, kz2 uv2) {
    const float *M = lod.camera_from_world;
    const kz3 pc = mk3(M[0] * p.x + M[1] * p.y + M[2] * p.z + M[3], M[4] * p.x + M[5] * p.y + M[6] * p.z + M[7], M[8] * p.x + M[9] * p.y + M[10] * p.z + M[11]);
    const kz3 nc = mk3(c2w[0] * n.x + c2w[4] * n.y + c2w[8] * n.z, c2w[1] * n.x + c2w[5] * n.y + c2w[9] * n.z, c2w[2] * n.x + c2w[6] * n.y + c2w[10] * n.z);
    /* RotateFromTo(normalize(pc), +z): the reflection pair through `refl` */
    const kz3 from = normalized(pc);
    const kz3 refl = fabsf(from.x) < 0.72f ? mk3(1.f, 0.f, 0.f) : (fabsf(from.y) < 0.72f ? mk3(0.f, 1.f, 0.f) : mk3(0.f, 0.f, 1.f));
    const kz3 u = refl - from, v = refl - mk3(0.f, 0.f, 1.f);
    const float uu = dot(u, u), vv = dot(v, v), uv = dot(u, v);
    const float a = 2.f / uu, b = 2.f / vv, c = 4.f * uv / (uu * vv);
    float R[9];
    const float uc[3] = {u.x, u.y, u.z}, vc[3] = {v.x, v.y, v.z};
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) R[3 * i + j] = (i == j ? 1.f : 0.f) - a * uc[i] * uc[j] - b * vc[i] * vc[j] + c * vc[i] * uc[j];
    auto rot = [&](kz3 w) { return mk3(R[0] * w.x + R[1] * w.y + R[2] * w.z, R[3] * w.x + R[4] * w.y + R[5] * w.z, R[6] * w.x + R[7] * w.y + R[8] * w.z); };
    auto rot_inv = [&](kz3 w) { return mk3(R[0] * w.x + R[3] * w.y + R[6] * w.z, R[1] * w.x + R[4] * w.y + R[7] * w.z, R[2] * w.x + R[5] * w.y + R[8] * w.z); };
    /* pbrt intersects the plane (pz, nz), pz = rot(pc) = (0, 0, |pc|), with the rays t * r and takes t * r - pz.  That difference is ~1e-3
     * of |pc| at a pixel's step, so it is formed here without the cancellation: pz is (0, 0, |pc|) exactly, and with nz.r = nz.z + e,
     * e = nz.x r.x + nz.y r.y + nz.z (r.z - 1), t - |pc| = -|pc| e / nz.r.  The same quantity, rounded to a few ulps instead of 1e-4. */
    const kz3 nz = rot(nc);
    const float pzz = norm(pc);
    auto offset = [&](const float *dd) {
        const kz3 r = mk3(dd[0], dd[1], 1.f + dd[2]);
        const float e = nz.x * dd[0] + nz.y * dd[1] + nz.z * dd[2];
        const float nr = dot(nz, r);
        const float t = nz.z * pzz / nr, t_minus = -pzz * e / nr;
        return rot_inv(mk3(t * r.x, t * r.y, t_minus + t * dd[2]));
    };
    const kz3 ox = offset(lod.ddx), oy = offset(lod.ddy);
    auto to_world_v = [&](kz3 w) { return mk3(c2w[0] * w.x + c2w[1] * w.y + c2w[2] * w.z, c2w[4] * w.x + c2w[5] * w.y + c2w[6] * w.z, c2w[8] * w.x + c2w[9] * w.y + c2w[10] * w.z); };
    const kz3 dpdx = lod.spp_scale * to_world_v(ox), dpdy = lod.spp_scale * to_world_v(oy);
    /* barycentric Jacobian of the triangle */
    const kz3 e1 = p1 - p0, e2 = p2 - p0;
    const float g11 = dot(e1, e1), g12 = dot(e1, e2), g22 = dot(e2, e2);
    float inv_det = 1.f / (g11 * g22 - g12 * g12);
    if (!isfinite(inv_det)) inv_det = 0.f;
    const kz2 du1 = mk2(uv1.x - uv0.x, uv1.y - uv0.y), du2 = mk2(uv2.x - uv0.x, uv2.y - uv0.y);
    auto map = [&](kz3 dp, float &duo, float &dvo) {
        const float r1 = dot(e1, dp), r2 = dot(e2, dp);
        const float b1 = (g22 * r1 - g12 * r2) * inv_det, b2 = (g11 * r2 - g12 * r1) * inv_det;
        duo = kz_lod_clamp(b1 * du1.x + b2 * du2.x);
        dvo = kz_lod_clamp(b1 * du1.y + b2 * du2.y);
    };
    KzUvDiff r;
    map(dpdx, r.dudx, r.dvdx);
    map(dpdy, r.dudy, r.dvdy);
    return r;
}
/* The footprint of hit `h` filled into `its` (fill_intersection): its triangle is read again (the sectors fill_intersection just read);
 * a mesh without uvs uses the barycentrics, as its.uv does.  Nothing of `its` but p, geo_n and the mesh is used: its.dpdu carries the
 * reference's quirks (only a positive uv determinant counts, a previous hit's value can carry over). */
KZ_HD KzUvDiff kz_its_footprint(const KzScene &sc, const KzTexLod &lod, const KzHit &h, const KzIts &its) {
    const KzMeshRec m = sc.meshes[h.geom];
    const KzU4 F = sc.indices[(size_t)m.index_offset + h.prim];
    const KzVertex v0 = kz_vertex(sc, m, F.x), v1 = kz_vertex(sc, m, F.y), v2 = kz_vertex(sc, m, F.z);
    const bool hasUV = (m.flags & KZ_MESH_HAS_UVS) != 0;
    const kz2 uv0 = hasUV ? kz_vuv(v0) : mk2(0.f, 0.f), uv1 = hasUV ? kz_vuv(v1) : mk2(1.f, 0.f), uv2 = hasUV ? kz_vuv(v2) : mk2(0.f, 1.f);
    return kz_uv_footprint(lod, sc.camera.camera_to_world, its.p, its.geo_n, kz_vpos(v0), kz_vpos(v1), kz_vpos(v2), uv0, uv1, uv2);
}

#endif
