/* kz_refit.cuh -- device side of kzgpu_accel_refit (the per-item arithmetic is in kz_refit.h).
 *
 *   k_refit_tris    every 48-byte triangle record re-gathered from the vertex records (kz_refit_tri), and max |coordinate| of all of
 *                   them into an ordered uint (as k_scene_bounds does): KzScene::scene_max_abs scales the traversal slack
 *   k_refit_check   per level, once per built accel: the internal children of level l lie in level l + 1 and the triangles of every node
 *                   in the record array -- what the bottom-up order and the reads of k_refit_level rely on
 *   k_refit_level   one launch per wide-tree level, deepest first: every node of [lo, hi) refitted (kz_refit_node) from the records and
 *                   the boxes its internal children left in `boxes` in the previous launch; no atomics
 */
#ifndef KZ_REFIT_CUH
#define KZ_REFIT_CUH
#include "kz_refit.h"
#include "kz_lbvh.cuh"

__global__ void k_refit_tris(const KzMeshRec *meshes, const KzVertex *vertices, const KzU4 *indices, KzF4 *tris, uint32_t n_tris, uint32_t *max_abs) {
    float m = 0.f;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_tris; i += gridDim.x * blockDim.x)
        m = fmaxf(m, kz_refit_tri(meshes, vertices, indices, tris, i));
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_down_sync(0xFFFFFFFFu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(max_abs, kzlbvh::f2ord(m));
}

__global__ void k_refit_check(const KzNode8 *nodes, uint32_t lo, uint32_t hi, uint32_t next_lo, uint32_t next_hi, uint32_t n_tris, uint32_t *bad) {
    bool b = false;
    for (uint32_t i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += gridDim.x * blockDim.x) {
        const uint4 w = reinterpret_cast<const uint4 *>(nodes + i)[0], x = reinterpret_cast<const uint4 *>(nodes + i)[1];
        const uint32_t imask = w.w >> 24, child_base = x.x, tri_base = x.y, trimask = x.z;
        if (imask) b |= child_base < next_lo || (uint64_t)child_base + __popc(imask) > next_hi;
        if (trimask) b |= (uint64_t)tri_base + __popc(trimask) > n_tris;
    }
    if (b) atomicOr(bad, 1u);
}

__global__ void k_refit_level(KzNode8 *nodes, const KzF4 *tris, KzBox *boxes, uint32_t lo, uint32_t hi) {
    for (uint32_t i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += gridDim.x * blockDim.x) {
        KzNode8 n = nodes[i];
        boxes[i] = kz_refit_node(n, tris, boxes);
        nodes[i] = n;
    }
}

#endif
