/* kz_ingest.cuh -- scene ingest and frame merge kernels (device side of kzgpu_scene_upload / kzgpu_render).
 *
 *   k_ingest_vertices   Mesh::m_V / m_N / m_UV (mesh.h:175-178: packed xyz / uv arrays) -> 32-byte KzVertex records
 *   k_update_vertices   kzgpu_mesh_update: new positions (and normals) into existing KzVertex records, the other fields kept
 *   k_transform_vertices kzgpu_mesh_transform: a mesh's rest pose placed by a matrix (kz_transform.h) into its KzVertex records, u / v kept
 *   k_copy_rest         positions (and normals) of KzVertex records -> a mesh's rest pose (packed xyz arrays)
 *   k_ingest_indices    Mesh::m_F -> 16-byte index records, validated against the vertex count
 *   k_ingest_texels     decoded rgb image -> float4 texels (level 0)
 *   k_gather_tris       (mesh table, vertex records, index records) -> the accel builders' triangle list in scene
 *                       order (Accel::addMesh order, accel.cpp:21-23,40-53: geomID = mesh index, primID = face index)
 *   k_frame_reduce      ImageBlock::put(ImageBlock&) (block.cpp:87-96) across the devices of a context: device g sums slice g
 *                       of every device's frame through peer (NVLink) loads and stores the result into the root's frame
 *
 * The raw arrays are copied into HBM as they are (one cudaMemcpyAsync per array, or read in place when the caller's
 * pointers already are device pointers); nothing of a mesh is touched element by element on the host.
 */
#ifndef KZ_INGEST_CUH
#define KZ_INGEST_CUH
#include "kz_scene.h"
#include "kz_bvh_build.h"
#include "kz_transform.h"

__global__ void k_ingest_vertices(const float *pos, const float *nrm, const float *uv, uint32_t n, KzVertex *out) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        KzVertex v;
        v.px = pos[3 * (size_t)i]; v.py = pos[3 * (size_t)i + 1]; v.pz = pos[3 * (size_t)i + 2];
        v.nx = nrm ? nrm[3 * (size_t)i] : 0.f; v.ny = nrm ? nrm[3 * (size_t)i + 1] : 0.f; v.nz = nrm ? nrm[3 * (size_t)i + 2] : 0.f;
        v.u = uv ? uv[2 * (size_t)i] : 0.f; v.v = uv ? uv[2 * (size_t)i + 1] : 0.f;
        float4 *o = reinterpret_cast<float4 *>(out + i);
        o[0] = make_float4(v.px, v.py, v.pz, v.u);
        o[1] = make_float4(v.nx, v.ny, v.nz, v.v);
    }
}

__global__ void k_update_vertices(const float *pos, const float *nrm, uint32_t n, KzVertex *out) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float4 *o = reinterpret_cast<float4 *>(out + i);
        const float4 a = o[0];
        o[0] = make_float4(pos[3 * (size_t)i], pos[3 * (size_t)i + 1], pos[3 * (size_t)i + 2], a.w);
        if (nrm) { const float4 b = o[1]; o[1] = make_float4(nrm[3 * (size_t)i], nrm[3 * (size_t)i + 1], nrm[3 * (size_t)i + 2], b.w); }
    }
}

/* rest_nrm == nullptr: the records' normals are kept (a mesh without normals) */
__global__ void k_transform_vertices(const float *rest_pos, const float *rest_nrm, uint32_t n, KzXform x, KzVertex *out) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float4 *o = reinterpret_cast<float4 *>(out + i);
        float r[3];
        kz_transform_point(x.m, rest_pos + 3 * (size_t)i, r);
        o[0] = make_float4(r[0], r[1], r[2], o[0].w);
        if (rest_nrm) {
            kz_transform_normal(x.inv, rest_nrm + 3 * (size_t)i, r);
            o[1] = make_float4(r[0], r[1], r[2], o[1].w);
        }
    }
}

/* nrm == nullptr: positions only */
__global__ void k_copy_rest(const KzVertex *v, uint32_t n, float *pos, float *nrm) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const KzVertex r = v[i];
        pos[3 * (size_t)i] = r.px; pos[3 * (size_t)i + 1] = r.py; pos[3 * (size_t)i + 2] = r.pz;
        if (nrm) { nrm[3 * (size_t)i] = r.nx; nrm[3 * (size_t)i + 1] = r.ny; nrm[3 * (size_t)i + 2] = r.nz; }
    }
}

/* bad[0] is set when an index is >= n_vertices (Mesh faces must reference existing vertices, mesh.cpp:296-318) */
__global__ void k_ingest_indices(const uint32_t *idx, uint32_t n_tris, uint32_t n_vertices, KzU4 *out, uint32_t *bad) {
    bool any_bad = false;
    for (uint32_t f = blockIdx.x * blockDim.x + threadIdx.x; f < n_tris; f += gridDim.x * blockDim.x) {
        const uint32_t a = idx[3 * (size_t)f], b = idx[3 * (size_t)f + 1], c = idx[3 * (size_t)f + 2];
        any_bad |= a >= n_vertices || b >= n_vertices || c >= n_vertices;
        reinterpret_cast<uint4 *>(out)[f] = make_uint4(a, b, c, 0u);
    }
    if (any_bad) atomicOr(bad, 1u);
}

__global__ void k_ingest_texels(const float *rgb, size_t n, KzF4 *out) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        reinterpret_cast<float4 *>(out)[i] = make_float4(rgb[3 * i], rgb[3 * i + 1], rgb[3 * i + 2], 1.f);
}

/* One thread per scene triangle; the owning mesh is found by bisection over the (ascending) index offsets. */
__global__ void k_gather_tris(const KzMeshRec *meshes, uint32_t n_meshes, const KzVertex *vertices, const KzU4 *indices, uint32_t n_tris, kzbvh::Tri *out) {
    for (uint32_t f = blockIdx.x * blockDim.x + threadIdx.x; f < n_tris; f += gridDim.x * blockDim.x) {
        uint32_t lo = 0u, hi = n_meshes;          /* last mesh with index_offset <= f (empty meshes share an offset: take the last) */
        while (hi - lo > 1u) { const uint32_t mid = (lo + hi) >> 1; if (meshes[mid].index_offset <= f) lo = mid; else hi = mid; }
        const KzMeshRec m = meshes[lo];
        const uint4 t = reinterpret_cast<const uint4 *>(indices)[f];
        const uint32_t vi[3] = {t.x, t.y, t.z};
        kzbvh::Tri r;
        for (int k = 0; k < 3; ++k) {
            const float4 p = reinterpret_cast<const float4 *>(vertices + m.vertex_offset + vi[k])[0];
            r.p[k][0] = p.x; r.p[k][1] = p.y; r.p[k][2] = p.z;
        }
        r.geom = lo; r.prim = f - m.index_offset;
        out[f] = r;
    }
}

#define KZ_MAX_DEVICES 16
struct KzFramePtrs { KzF4 *f[KZ_MAX_DEVICES]; };

/* Runs on every device of a multi-device context once all of them finished splatting: this device sums texels [begin, end) of
 * all n frames (its own from HBM, the others through NVLink peer loads) and writes the sums into the root's frame (a peer store
 * unless this device is the root).  Every texel of the root's frame is written by exactly one device, and a texel is read
 * before it is overwritten by the same thread, so the merge is in place; the inbound traffic of the root is (n-1)/n of ONE frame
 * instead of n-1 frames. */
__global__ void k_frame_reduce(KzFramePtrs frames, int n, size_t begin, size_t end) {
    for (size_t i = begin + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < end; i += (size_t)gridDim.x * blockDim.x) {
        float4 acc = __ldcg(reinterpret_cast<const float4 *>(frames.f[0]) + i);
        for (int g = 1; g < n; ++g) {
            const float4 v = __ldcg(reinterpret_cast<const float4 *>(frames.f[g]) + i);
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
        __stcg(reinterpret_cast<float4 *>(frames.f[0]) + i, acc);
    }
}

#endif
