/* kz_host_scene.h -- flattens a kz_scene_desc into the contiguous arrays of kz_scene.h on the
 * host.  kz_api.cu uploads each array to HBM and patches the pointers; tests/hostemu points a
 * KzScene straight at the host vectors.  Reference counterparts: Scene::activate light list
 * (scene.cpp:42-46), Mesh::activate area CDF (mesh.cpp:24-45, dpdf.h:35-81), PMJ02BN pixel
 * sample buckets (sampler.cpp:290-314). */
#ifndef KZ_HOST_SCENE_H
#define KZ_HOST_SCENE_H
#include "kz_scene.h"
#include "kz_bvh_build.h"
#include <string>
#include <vector>

struct KzHostScene {
    std::vector<KzMeshRec> meshes;
    std::vector<KzVertex> vertices;
    std::vector<float> light_cdf;
    std::vector<KzU4> indices;
    std::vector<int32_t> light_meshes;
    std::vector<float> light_bounds;    /* per emitter (light_meshes order): lo[3], hi[3] of its vertices */
    std::vector<kz_bsdf_desc> bsdfs;
    std::vector<kz_texture_desc> textures;
    std::vector<KzImageRec> images;
    std::vector<KzF4> texels;
    std::vector<kz_light_desc> lights;
    std::vector<uint16_t> blue_noise;
    std::vector<uint32_t> pmj;
    std::vector<kz2> pmj_pixel_samples;
    std::vector<kzbvh::Tri> tris;       /* scene order, input of the accel build */
    KzScene sc;                         /* pointers into the vectors above once finalize() ran */
    uint64_t total_vertices = 0, total_triangles = 0;
    std::string error;

    /* geometry = true: vertex / index records and the triangle list are built here (tests/hostemu runs the device headers on
     * these vectors).  geometry = false (kz_api.cu): only the small tables are built; the mesh arrays go to HBM as they are and
     * the records are made there (kz_ingest.cuh), so `vertices`, `indices` and `tris` stay empty and indices are validated on
     * the device.  Light meshes need host-readable positions / indices in both modes (area CDF, mesh.cpp:24-45). */
    bool flatten(const kz_scene_desc *d, bool geometry = true) {
        memset(&sc, 0, sizeof(sc));
        if (!d) { error = "null scene"; return false; }
        if (d->n_meshes && !d->meshes) { error = "meshes missing"; return false; }
        bsdfs.assign(d->bsdfs, d->bsdfs + d->n_bsdfs);
        textures.assign(d->textures, d->textures + d->n_textures);
        lights.assign(d->lights, d->lights + d->n_lights);
        for (uint32_t i = 0; i < d->n_bsdfs; ++i) {
            const kz_bsdf_desc &b = d->bsdfs[i];
            auto texok = [&](int t) { return t >= 0 && t < (int)d->n_textures; };
            if (b.type == KZ_BSDF_KISS) {
                if (!texok(b.base_color) || !texok(b.roughness) || !texok(b.metallic)) { error = "kazenstandard needs baseColor/roughness/metallic textures"; return false; }
            } else if (b.type == KZ_BSDF_NORMALMAP) {
                if (!texok(b.normal_map) || b.nested < 0 || b.nested >= (int)d->n_bsdfs) { error = "normalmap needs a texture and a nested bsdf"; return false; }
                if (d->bsdfs[b.nested].type == KZ_BSDF_NORMALMAP) { error = "nested normalmap is unsupported"; return false; }
            } else if (b.type == KZ_BSDF_LAMBERTIAN || b.type == KZ_BSDF_GGX) {
                if (!texok(b.base_color)) { error = "lambertian / ggx need an albedo texture"; return false; }
            } else if (b.type < KZ_BSDF_DIFFUSE || b.type > KZ_BSDF_ROUGHDIELECTRIC) { error = "bsdf type outside the hot-path scope"; return false; }
        }
        for (uint32_t i = 0; i < d->n_textures; ++i) {
            const kz_texture_desc &t = d->textures[i];
            if (t.type == KZ_TEX_IMAGE && (t.image < 0 || t.image >= (int)d->n_images)) { error = "image index out of range"; return false; }
            for (int c = 0; c < 3; ++c) if (t.child[c] >= (int)d->n_textures || t.child[c] < -1) { error = "texture child out of range"; return false; }
        }
        /* expression trees are evaluated with a fixed-depth stack on the device (kz_tex_eval_tree): reject what it cannot hold */
        for (uint32_t i = 0; i < d->n_textures; ++i) {
            const int depth = textureDepth(d, (int)i, 0);
            if (depth < 0) { error = "texture graph has a cycle"; return false; }
            if (depth > KZ_TEX_MAX_DEPTH_HOST) { error = "texture tree deeper than " + std::to_string(KZ_TEX_MAX_DEPTH_HOST) + " levels is unsupported"; return false; }
        }
        /* images: level 0 as float4 texels followed by room for the mip pyramid (filled on the GPU by k_mip_level) */
        for (uint32_t i = 0; i < d->n_images; ++i) {
            const kz_image_desc &im = d->images[i];
            if (im.width <= 0 || im.height <= 0 || !im.rgb) { error = "bad image"; return false; }
            if (im.width > 65536 || im.height > 65536) { error = "image larger than 65536 texels per side"; return false; }
            /* level 0 only: ImageTexture::eval passes zero derivatives to OIIO (texture.cpp:52-57), which resolves to the finest
             * level; the pyramid is built on demand by kzgpu_image_lookup (n_levels stays 0 for the renderer) */
            KzImageRec r; r.width = im.width; r.height = im.height; r.texel_offset = (uint32_t)total_texels; r.n_levels = 0;
            const size_t n = (size_t)im.width * im.height;
            if (total_texels + n > 0xFFFFFFFFull) { error = "texture atlas larger than 2^32 texels"; return false; }
            total_texels += n;
            if (geometry) {
                texels.resize(total_texels, KzF4{0.f, 0.f, 0.f, 0.f});
                for (size_t k = 0; k < n; ++k) {
                    KzF4 &t = texels[r.texel_offset + k];
                    t.x = im.rgb[3 * k]; t.y = im.rgb[3 * k + 1]; t.z = im.rgb[3 * k + 2]; t.w = 1.f;
                }
            }
            images.push_back(r);
        }
        uint64_t voff = 0, foff = 0;
        sc.n_invisible_lights = 0;
        for (uint32_t g = 0; g < d->n_meshes; ++g) {
            const kz_mesh_desc &m = d->meshes[g];
            if (!m.positions || !m.indices) { error = "mesh buffers missing"; return false; }
            if (m.bsdf < 0 || m.bsdf >= (int)d->n_bsdfs) { error = "mesh bsdf index out of range"; return false; }
            if (m.light >= (int)d->n_lights) { error = "mesh light index out of range"; return false; }
            KzMeshRec r; memset(&r, 0, sizeof(r));
            if (voff + m.n_vertices > 0xFFFFFFFFull || foff + m.n_triangles > 0x7FFFFFFFull) { error = "scene larger than 2^32 vertices / 2^31 triangles"; return false; }
            r.vertex_offset = (uint32_t)voff; r.index_offset = (uint32_t)foff; r.n_triangles = m.n_triangles;
            r.bsdf = m.bsdf; r.light = m.light;
            r.flags = (m.normals ? KZ_MESH_HAS_NORMALS : 0u) | (m.uvs ? KZ_MESH_HAS_UVS : 0u);
            if (geometry) vertices.reserve(vertices.size() + m.n_vertices);
            for (uint32_t i = 0; geometry && i < m.n_vertices; ++i) {
                KzVertex v; memset(&v, 0, sizeof(v));
                v.px = m.positions[3 * (size_t)i]; v.py = m.positions[3 * (size_t)i + 1]; v.pz = m.positions[3 * (size_t)i + 2];
                if (m.normals) { v.nx = m.normals[3 * (size_t)i]; v.ny = m.normals[3 * (size_t)i + 1]; v.nz = m.normals[3 * (size_t)i + 2]; }
                if (m.uvs) { v.u = m.uvs[2 * (size_t)i]; v.v = m.uvs[2 * (size_t)i + 1]; }
                vertices.push_back(v);
            }
            if (geometry) indices.reserve(indices.size() + m.n_triangles);
            for (uint32_t f = 0; geometry && f < m.n_triangles; ++f) {
                KzU4 t; t.x = m.indices[3 * (size_t)f]; t.y = m.indices[3 * (size_t)f + 1]; t.z = m.indices[3 * (size_t)f + 2]; t.w = 0u;
                if (t.x >= m.n_vertices || t.y >= m.n_vertices || t.z >= m.n_vertices) { error = "vertex index out of range"; return false; }
                indices.push_back(t);
            }
            if (m.light >= 0) {
                /* an emitter without triangles cannot be sampled (DiscretePDF over nothing, mesh.cpp:108-133) */
                if (m.n_triangles == 0) { error = "emissive mesh without triangles"; return false; }
                for (uint32_t f = 0; !geometry && f < m.n_triangles; ++f)
                    if (m.indices[3 * (size_t)f] >= m.n_vertices || m.indices[3 * (size_t)f + 1] >= m.n_vertices || m.indices[3 * (size_t)f + 2] >= m.n_vertices) { error = "vertex index out of range"; return false; }
                r.flags |= KZ_MESH_IS_LIGHT;
                if (d->lights[m.light].primary_visibility) r.flags |= KZ_MESH_LIGHT_VISIBLE;
                else ++sc.n_invisible_lights;
                r.cdf_offset = (uint32_t)light_cdf.size();
                light_cdf.resize(light_cdf.size() + m.n_triangles + 1);
                light_bounds.resize(light_bounds.size() + 6);
                emitter_tables(m.positions, m.indices, m.n_triangles, light_cdf.data() + r.cdf_offset, r.inv_area, light_bounds.data() + light_bounds.size() - 6);
                light_meshes.push_back((int32_t)g);
            }
            for (uint32_t f = 0; geometry && f < m.n_triangles; ++f) {
                kzbvh::Tri t;
                for (int k = 0; k < 3; ++k) {
                    const float *p = m.positions + 3 * (size_t)m.indices[3 * f + k];
                    t.p[k][0] = p[0]; t.p[k][1] = p[1]; t.p[k][2] = p[2];
                }
                t.geom = g; t.prim = f;
                tris.push_back(t);
            }
            meshes.push_back(r);
            voff += m.n_vertices; foff += m.n_triangles;
        }
        total_vertices = voff; total_triangles = foff;
        invisible_light_bounds();
        sc.n_meshes = d->n_meshes;
        sc.n_light_meshes = (int32_t)light_meshes.size();
        sc.background = d->background;
        if (sc.background >= (int)d->n_textures) { error = "background texture out of range"; return false; }
        sc.camera = d->camera;
        sc.integrator = d->integrator;
        if (sc.integrator.type < KZ_INTEGRATOR_PATH_MIS || sc.integrator.type > KZ_INTEGRATOR_PATH_MATS) { error = "unknown integrator type"; return false; }
        sc.filter = d->filter;
        sc.border = (int32_t)ceilf(d->filter.radius - 0.5f);
        sc.sampler_type = d->sampler.type;
        sc.sample_count = d->sampler.sample_count;
        sc.seed = d->sampler.seed;
        sc.res_x = d->sampler.res_x; sc.res_y = d->sampler.res_y;
        if (sc.camera.width <= 0 || sc.camera.height <= 0 || sc.camera.width > 65535 || sc.camera.height > 65535) { error = "camera size out of range"; return false; }
        if (!(d->filter.radius > 0.f) || d->filter.radius > 7.f) { error = "filter radius out of range"; return false; }
        if (sc.sample_count == 0) { error = "sample_count is zero"; return false; }
        if (sc.sampler_type == KZ_SAMPLER_PMJ02BN) {
            if (!d->sampler.blue_noise || !d->sampler.pmj02bn) { error = "pmj02bn needs the blue-noise and pmj02bn tables (see kzgpu_fallback_tables)"; return false; }
            blue_noise.assign(d->sampler.blue_noise, d->sampler.blue_noise + 48 * 128 * 128);
            pmj.assign(d->sampler.pmj02bn, d->sampler.pmj02bn + 5 * 65536 * 2);
            if (sc.sample_count > 65536) sc.sample_count = 65536;
            buildPmjPixelSamples();
        }
        finalize();
        return true;
    }

    /* Mesh::activate + DiscretePDF::normalize (mesh.cpp:24-45, dpdf.h:35-81) for an emitter of n_triangles > 0 triangles: its area CDF
     * (n_triangles + 1 floats from 0 to 1), the normalisation 1 / sum(area) and the bounds of the vertices its triangles use.
     * kzgpu_scene_upload (through flatten) and kzgpu_mesh_update both come here, so an updated emitter samples as a freshly uploaded one. */
    static void emitter_tables(const float *positions, const uint32_t *idx, uint32_t n_triangles, float *cdf, float &inv_area, float *bounds) {
        for (int a = 0; a < 3; ++a) { bounds[a] = kz_u2f(0x7f800000u); bounds[3 + a] = kz_u2f(0xff800000u); }
        cdf[0] = 0.0f;
        for (uint32_t f = 0; f < n_triangles; ++f) {
            const float *p0 = positions + 3 * (size_t)idx[3 * (size_t)f], *p1 = positions + 3 * (size_t)idx[3 * (size_t)f + 1],
                        *p2 = positions + 3 * (size_t)idx[3 * (size_t)f + 2];
            for (const float *q : {p0, p1, p2})
                for (int a = 0; a < 3; ++a) { bounds[a] = fminf(bounds[a], q[a]); bounds[3 + a] = fmaxf(bounds[3 + a], q[a]); }
            kz3 e1 = mk3(kz_sub(p1[0], p0[0]), kz_sub(p1[1], p0[1]), kz_sub(p1[2], p0[2]));
            kz3 e2 = mk3(kz_sub(p2[0], p0[0]), kz_sub(p2[1], p0[1]), kz_sub(p2[2], p0[2]));
            kz3 c = mk3(kz_sub(kz_mul(e1.y, e2.z), kz_mul(e1.z, e2.y)), kz_sub(kz_mul(e1.z, e2.x), kz_mul(e1.x, e2.z)),
                        kz_sub(kz_mul(e1.x, e2.y), kz_mul(e1.y, e2.x)));
            float n2 = kz_add(kz_add(kz_mul(c.x, c.x), kz_mul(c.y, c.y)), kz_mul(c.z, c.z));
            float area = kz_mul(0.5f, kz_sqrt(n2));
            cdf[f + 1] = kz_add(cdf[f], area);
        }
        const float sum = cdf[n_triangles];
        if (sum > 0) {
            inv_area = kz_div(1.0f, sum);
            for (uint32_t k = 1; k <= n_triangles; ++k) cdf[k] = kz_mul(cdf[k], inv_area);
            cdf[n_triangles] = 1.0f;
        } else inv_area = 0.f;
    }

    /* sc.inv_light_lo / hi: the bounds of the invisible emitters' vertices (shadow rays stop early outside them, KzWalk::settles) */
    void invisible_light_bounds() {
        for (int a = 0; a < 3; ++a) { sc.inv_light_lo[a] = kz_u2f(0x7f800000u); sc.inv_light_hi[a] = kz_u2f(0xff800000u); }
        for (size_t k = 0; k < light_meshes.size(); ++k) {
            if (meshes[(size_t)light_meshes[k]].flags & KZ_MESH_LIGHT_VISIBLE) continue;
            for (int a = 0; a < 3; ++a) {
                sc.inv_light_lo[a] = fminf(sc.inv_light_lo[a], light_bounds[6 * k + a]);
                sc.inv_light_hi[a] = fmaxf(sc.inv_light_hi[a], light_bounds[6 * k + 3 + a]);
            }
        }
    }

    size_t total_texels = 0;
    enum { KZ_TEX_MAX_DEPTH_HOST = 4 };      /* == KZ_TEX_MAX_DEPTH of kz_shade.h */
    /* nodes on the longest root-to-leaf chain below `node`, -1 if a cycle is reachable */
    static int textureDepth(const kz_scene_desc *d, int node, int guard) {
        if (guard > 64) return -1;
        int deepest = 0;
        for (int c = 0; c < 3; ++c) {
            const int ch = d->textures[node].child[c];
            if (ch < 0) continue;
            const int sub = textureDepth(d, ch, guard + 1);
            if (sub < 0) return -1;
            deepest = std::max(deepest, sub);
        }
        return deepest + 1;
    }

    /* sampler.cpp:290-314 */
    void buildPmjPixelSamples() {
        auto log2i = [](int v) { int r = 0; while (v > 1) { v >>= 1; ++r; } return r; };
        auto isPow4 = [](int n) { if (n <= 0) return false; int x = (int)sqrt((double)n); if (x * x != n) return false; return !(n & (n - 1)); };
        int spp = (int)sc.sample_count;
        int up = isPow4(spp) ? spp : (1 << (2 * (1 + log2i(spp) / 2)));
        int tile = 1 << (8 - log2i(up) / 2);
        sc.pmj_tile_size = tile;
        pmj_pixel_samples.assign((size_t)tile * tile * spp, mk2(0.f, 0.f));
        std::vector<int> nStored((size_t)tile * tile, 0);
        for (int i = 0; i < 65536; ++i) {
            float x = (float)(pmj[(size_t)i * 2] * 0x1p-32), y = (float)(pmj[(size_t)i * 2 + 1] * 0x1p-32);
            x = kz_mul(x, (float)tile); y = kz_mul(y, (float)tile);
            int off = int(x) + int(y) * tile;
            if (nStored[off] == spp) continue;
            pmj_pixel_samples[(size_t)off * spp + nStored[off]] = mk2(kz_sub(x, floorf(x)), kz_sub(y, floorf(y)));
            ++nStored[off];
        }
    }

    void finalize() {
        sc.meshes = meshes.data();
        sc.vertices = vertices.data();
        sc.indices = indices.data(); sc.light_cdf = light_cdf.data(); sc.light_meshes = light_meshes.data();
        sc.bsdfs = bsdfs.data(); sc.textures = textures.data(); sc.images = images.data(); sc.texels = texels.data();
        sc.lights = lights.data();
        sc.blue_noise = blue_noise.data(); sc.pmj02bn = pmj.data(); sc.pmj_pixel_samples = pmj_pixel_samples.data();
    }
};

#endif
