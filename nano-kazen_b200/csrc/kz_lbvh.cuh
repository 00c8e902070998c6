/* kz_lbvh.cuh -- on-GPU accel build (replaces the Embree build of Accel::build, accel.cpp:25-61).
 *
 *   k_scene_bounds   centroid bounds + max |coordinate|           (block reduce + ordered-int atomics)
 *   k_morton         63-bit Morton key of every triangle centroid
 *   cub radix sort   (key, triangle) pairs  -- library utility, the only non-hand-written step
 *   k_karras         binary radix tree over the sorted keys (Karras 2012), one thread per internal node
 *   k_fit            bottom-up AABB fit, second-arriver-continues
 *   k_collapse       level-synchronous collapse into the 80-byte 8-wide compressed nodes of
 *                    kz_scene.h: subtrees of <= 3 triangles become leaf slots, the child with the
 *                    largest area is opened until 8 slots are used, slots are octant-ordered,
 *                    child boxes are quantised outwards in double precision (conservative).
 *
 * Tree quality does not affect results: culling is conservative and ties on t are broken by
 * (geomID, primID) in the traversal, so the host-SAH and the LBVH accel return identical hits.
 */
#ifndef KZ_LBVH_CUH
#define KZ_LBVH_CUH
#include "kz_scene.h"
#include "kz_bvh_build.h"
#include "kz_owner.h"
#include <cub/device/device_radix_sort.cuh>
#include <cuda_runtime.h>
#include <string>
#include <vector>

namespace kzlbvh {

struct Result {
    DevMem nodes, tris;          /* KzNode8[n_nodes] (allocated for more), KzF4[3 * n_tris] */
    uint32_t n_nodes = 0, n_tris = 0;
    float max_abs = 0.f;
    uint64_t launches = 0;
    int depth = 0;               /* wide-tree levels */
    std::vector<uint32_t> level_first;   /* level l = nodes [level_first[l], level_first[l + 1]) (kzgpu_accel_refit) */
};

struct Box6 { float lo[3], hi[3]; };

struct BuildState {
    const kzbvh::Tri *tris;      /* scene order */
    const float4 *rlo, *rhi;     /* pre-split references (nullptr: one reference per triangle): box lo | triangle index, box hi */
    uint32_t n;                  /* references */
    const uint32_t *order;       /* sorted position -> triangle */
    const unsigned long long *keys;
    int32_t *left, *right;       /* >= 0 internal node, < 0: ~leaf (sorted position) */
    int32_t *parent;             /* [0, n-1): internal nodes, [n-1, 2n-1): leaves */
    uint32_t *first, *last;      /* sorted range covered by an internal node */
    KzF4 *blo, *bhi;             /* internal node boxes */
    uint32_t *flags;
};

__device__ __forceinline__ uint32_t f2ord(float f) { uint32_t u = __float_as_uint(f); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); }
__host__ __device__ __forceinline__ float ord2f(uint32_t u) {
    u = (u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u;
#if defined(__CUDA_ARCH__)
    return __uint_as_float(u);
#else
    float f; memcpy(&f, &u, 4); return f;
#endif
}

/* bounds[0..2] = min centroid, [3..5] = max centroid, [6] = max |coordinate| (all as ordered uints) */
__global__ void k_scene_bounds(const kzbvh::Tri *tris, uint32_t n, uint32_t *bounds) {
    float lo[3] = {3.4e38f, 3.4e38f, 3.4e38f}, hi[3] = {-3.4e38f, -3.4e38f, -3.4e38f}, mabs = 0.f;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const kzbvh::Tri t = tris[i];
        for (int a = 0; a < 3; ++a) {
            const float mn = fminf(t.p[0][a], fminf(t.p[1][a], t.p[2][a])), mx = fmaxf(t.p[0][a], fmaxf(t.p[1][a], t.p[2][a]));
            const float c = 0.5f * (mn + mx);
            lo[a] = fminf(lo[a], c); hi[a] = fmaxf(hi[a], c);
            mabs = fmaxf(mabs, fmaxf(fabsf(mn), fabsf(mx)));
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        for (int a = 0; a < 3; ++a) {
            lo[a] = fminf(lo[a], __shfl_down_sync(0xFFFFFFFFu, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_down_sync(0xFFFFFFFFu, hi[a], o));
        }
        mabs = fmaxf(mabs, __shfl_down_sync(0xFFFFFFFFu, mabs, o));
    }
    if ((threadIdx.x & 31) == 0) {
        for (int a = 0; a < 3; ++a) { atomicMin(bounds + a, f2ord(lo[a])); atomicMax(bounds + 3 + a, f2ord(hi[a])); }
        atomicMax(bounds + 6, f2ord(mabs));
    }
}

__device__ __forceinline__ unsigned long long expand21(unsigned long long v) {
    v &= 0x1FFFFFull;
    v = (v | (v << 32)) & 0x1F00000000FFFFull;
    v = (v | (v << 16)) & 0x1F0000FF0000FFull;
    v = (v | (v << 8)) & 0x100F00F00F00F00Full;
    v = (v | (v << 4)) & 0x10C30C30C30C30C3ull;
    v = (v | (v << 2)) & 0x1249249249249249ull;
    return v;
}

__global__ void k_morton(const kzbvh::Tri *tris, const float4 *rlo, const float4 *rhi, uint32_t n, const uint32_t *bounds, unsigned long long *keys, uint32_t *vals) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float blo[3], bhi[3];
    if (rlo) {
        const float4 l = rlo[i], h = rhi[i];
        blo[0] = l.x; blo[1] = l.y; blo[2] = l.z; bhi[0] = h.x; bhi[1] = h.y; bhi[2] = h.z;
    } else {
        const kzbvh::Tri t = tris[i];
        for (int a = 0; a < 3; ++a) { blo[a] = fminf(t.p[0][a], fminf(t.p[1][a], t.p[2][a])); bhi[a] = fmaxf(t.p[0][a], fmaxf(t.p[1][a], t.p[2][a])); }
    }
    unsigned long long code = 0ull;
    for (int a = 0; a < 3; ++a) {
        const float lo = ord2f(bounds[a]), hi = ord2f(bounds[3 + a]);
        const float mn = blo[a], mx = bhi[a];
        const float c = 0.5f * (mn + mx);
        const float ext = hi - lo;
        float u = ext > 0.f ? (c - lo) / ext : 0.f;
        u = fminf(fmaxf(u, 0.f), 1.f);
        unsigned long long q = (unsigned long long)(u * 2097152.0f);
        if (q > 2097151ull) q = 2097151ull;
        code |= expand21(q) << (2 - a);
    }
    keys[i] = code; vals[i] = i;
}

__device__ __forceinline__ int kz_delta(const unsigned long long *keys, int n, int i, int j) {
    if (j < 0 || j >= n) return -1;
    const unsigned long long a = keys[i], b = keys[j];
    if (a == b) return 64 + __clz(i ^ j);
    return __clzll((long long)(a ^ b));
}

__global__ void k_karras(BuildState b) {
    const int n = (int)b.n;
    const int i = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (i >= n - 1) return;
    const unsigned long long *keys = b.keys;
    const int d = (kz_delta(keys, n, i, i + 1) - kz_delta(keys, n, i, i - 1)) >= 0 ? 1 : -1;
    const int dmin = kz_delta(keys, n, i, i - d);
    int lmax = 2;
    while (kz_delta(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int t = lmax >> 1; t >= 1; t >>= 1)
        if (kz_delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
    const int j = i + l * d;
    const int dnode = kz_delta(keys, n, i, j);
    int s = 0;
    for (int div = 2;; div <<= 1) {
        const int t = (l + div - 1) / div;
        if (kz_delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
        if (t <= 1) break;
    }
    const int gamma = i + s * d + (d < 0 ? -1 : 0);
    const int lo = i < j ? i : j, hi = i < j ? j : i;
    const int lc = (lo == gamma) ? ~gamma : gamma;
    const int rc = (hi == gamma + 1) ? ~(gamma + 1) : (gamma + 1);
    b.left[i] = lc; b.right[i] = rc;
    b.first[i] = (uint32_t)lo; b.last[i] = (uint32_t)hi;
    b.parent[lc >= 0 ? lc : (n - 1 + ~lc)] = i;
    b.parent[rc >= 0 ? rc : (n - 1 + ~rc)] = i;
    if (i == 0) b.parent[0] = -1;
}

__device__ __forceinline__ Box6 tri_box(const kzbvh::Tri &t) {
    Box6 r;
    for (int a = 0; a < 3; ++a) {
        r.lo[a] = fminf(t.p[0][a], fminf(t.p[1][a], t.p[2][a]));
        r.hi[a] = fmaxf(t.p[0][a], fmaxf(t.p[1][a], t.p[2][a]));
    }
    return r;
}
__device__ __forceinline__ uint32_t ref_tri(const BuildState &b, uint32_t ref) { return b.rlo ? __float_as_uint(b.rlo[ref].w) : ref; }
__device__ __forceinline__ Box6 child_box(const BuildState &b, int c) {
    if (c < 0) {
        const uint32_t ref = b.order[~c];
        if (!b.rlo) return tri_box(b.tris[ref]);
        const float4 l = b.rlo[ref], h = b.rhi[ref];
        Box6 r; r.lo[0] = l.x; r.lo[1] = l.y; r.lo[2] = l.z; r.hi[0] = h.x; r.hi[1] = h.y; r.hi[2] = h.z;
        return r;
    }
    /* ld.cg: boxes are produced by other SMs in the same launch (k_fit); never trust L1 here */
    const float4 lo = __ldcg(reinterpret_cast<const float4 *>(b.blo) + c), hi = __ldcg(reinterpret_cast<const float4 *>(b.bhi) + c);
    Box6 r; r.lo[0] = lo.x; r.lo[1] = lo.y; r.lo[2] = lo.z; r.hi[0] = hi.x; r.hi[1] = hi.y; r.hi[2] = hi.z;
    return r;
}

__global__ void k_fit(BuildState b) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= b.n) return;
    int node = b.parent[b.n - 1 + i];
    while (node >= 0) {
        __threadfence();
        if (atomicAdd(b.flags + node, 1u) == 0u) return;      /* first arriver leaves */
        __threadfence();
        const Box6 l = child_box(b, b.left[node]), r = child_box(b, b.right[node]);
        KzF4 lo, hi;
        lo.x = fminf(l.lo[0], r.lo[0]); lo.y = fminf(l.lo[1], r.lo[1]); lo.z = fminf(l.lo[2], r.lo[2]); lo.w = 0.f;
        hi.x = fmaxf(l.hi[0], r.hi[0]); hi.y = fmaxf(l.hi[1], r.hi[1]); hi.z = fmaxf(l.hi[2], r.hi[2]); hi.w = 0.f;
        __stcg(reinterpret_cast<float4 *>(b.blo) + node, make_float4(lo.x, lo.y, lo.z, 0.f));
        __stcg(reinterpret_cast<float4 *>(b.bhi) + node, make_float4(hi.x, hi.y, hi.z, 0.f));
        node = b.parent[node];
    }
}

#ifndef KZ_LBVH_MAXLEAF
#define KZ_LBVH_MAXLEAF 1u       /* triangles per leaf slot of the collapsed LBVH (1..3); measured on the 2^20-triangle soup: 1 -> 2146/1750, 2 -> 1999/1559, 3 -> 1905/1444 Mrays/s (every triangle gets its own child box) */
#endif
struct WorkItem { int32_t bnode; uint32_t wnode; };

struct CollapseState {
    BuildState b;
    KzNode8 *nodes;
    KzF4 *tris;
    uint32_t *node_counter, *tri_counter;
    const WorkItem *in;
    WorkItem *out;
    const uint32_t *in_count;    /* work items of this level (written by the previous level's launch) */
    uint32_t *out_count;         /* work items of the next level */
};

__device__ __forceinline__ uint32_t sub_count(const BuildState &b, int c) { return c < 0 ? 1u : b.last[c] - b.first[c] + 1u; }
__device__ __forceinline__ float box_area(const Box6 &x) {
    const float dx = x.hi[0] - x.lo[0], dy = x.hi[1] - x.lo[1], dz = x.hi[2] - x.lo[2];
    return 2.f * (dx * dy + dy * dz + dz * dx);
}

/* One launch per wide-tree level.  The level's item count lives in HBM (written by the previous launch), so the host enqueues
 * all levels back to back without reading anything back. */
__global__ void __launch_bounds__(64) k_collapse(CollapseState cs) {
    const uint32_t n_in = *cs.in_count;
    for (uint32_t wi = blockIdx.x * blockDim.x + threadIdx.x; wi < n_in; wi += gridDim.x * blockDim.x) {
    const BuildState &b = cs.b;
    const WorkItem it = cs.in[wi];
    int ch[8]; Box6 bx[8]; int nch = 0;
    const int root = it.bnode;
    if (root < 0 || sub_count(b, root) <= KZ_LBVH_MAXLEAF) { ch[0] = root; bx[0] = child_box(b, root); nch = 1; }
    else {
        ch[0] = b.left[root]; ch[1] = b.right[root];
        bx[0] = child_box(b, ch[0]); bx[1] = child_box(b, ch[1]); nch = 2;
    }
    while (nch < 8) {
        int best = -1; float bestA = -1.f;
        for (int i = 0; i < nch; ++i) {
            if (ch[i] < 0 || sub_count(b, ch[i]) <= KZ_LBVH_MAXLEAF) continue;
            const float a = box_area(bx[i]);
            if (a > bestA) { bestA = a; best = i; }
        }
        if (best < 0) break;
        const int c = ch[best];
        ch[best] = b.left[c]; bx[best] = child_box(b, ch[best]);
        ch[nch] = b.right[c]; bx[nch] = child_box(b, ch[nch]);
        ++nch;
    }
    Box6 nb;
    for (int a = 0; a < 3; ++a) { nb.lo[a] = 3.4e38f; nb.hi[a] = -3.4e38f; }
    for (int i = 0; i < nch; ++i)
        for (int a = 0; a < 3; ++a) { nb.lo[a] = fminf(nb.lo[a], bx[i].lo[a]); nb.hi[a] = fmaxf(nb.hi[a], bx[i].hi[a]); }
    /* slot assignment: greedy max of sum_a sign_s(a) * (child centre - node centre) */
    const float cen[3] = {0.5f * (nb.lo[0] + nb.hi[0]), 0.5f * (nb.lo[1] + nb.hi[1]), 0.5f * (nb.lo[2] + nb.hi[2])};
    int childAt[8]; for (int s = 0; s < 8; ++s) childAt[s] = -1;
    {
        uint32_t usedSlots = 0u, doneCh = 0u;
        for (int k = 0; k < nch; ++k) {
            int bi = -1, bs = -1; float bc = -3.4e38f;
            for (int i = 0; i < nch; ++i) {
                if (doneCh & (1u << i)) continue;
                const float dx = 0.5f * (bx[i].lo[0] + bx[i].hi[0]) - cen[0], dy = 0.5f * (bx[i].lo[1] + bx[i].hi[1]) - cen[1],
                            dz = 0.5f * (bx[i].lo[2] + bx[i].hi[2]) - cen[2];
                for (int s = 0; s < 8; ++s) {
                    if (usedSlots & (1u << s)) continue;
                    const float c = ((s & 1) ? dx : -dx) + ((s & 2) ? dy : -dy) + ((s & 4) ? dz : -dz);
                    if (c > bc) { bc = c; bi = i; bs = s; }
                }
            }
            childAt[bs] = bi; usedSlots |= 1u << bs; doneCh |= 1u << bi;
        }
    }
    /* quantisation frame: smallest power of two e with ceil(ext / 2^e) <= 255 */
    int e[3];
    for (int a = 0; a < 3; ++a) {
        const double ext = (double)nb.hi[a] - (double)nb.lo[a];
        int ee = 1 - 127;
        if (ext > 0.0) { frexp(ext / 255.0, &ee); }
        int biased = ee + 127;
        biased = biased < 1 ? 1 : (biased > 254 ? 254 : biased);
        while (biased < 254 && ceil(ext / ldexp(1.0, biased - 127)) > 255.0) ++biased;
        e[a] = biased;
    }
    uint32_t n_internal = 0, n_tris = 0;
    for (int s = 0; s < 8; ++s) {
        if (childAt[s] < 0) continue;
        const int c = ch[childAt[s]];
        const uint32_t cnt = sub_count(b, c);
        if (c >= 0 && cnt > KZ_LBVH_MAXLEAF) ++n_internal; else n_tris += cnt;
    }
    const uint32_t child_base = n_internal ? atomicAdd(cs.node_counter, n_internal) : 0u;
    const uint32_t tri_base = n_tris ? atomicAdd(cs.tri_counter, n_tris) : 0u;
    const uint32_t out_base = n_internal ? atomicAdd(cs.out_count, n_internal) : 0u;

    KzNode8 nd;
    memset(&nd, 0, sizeof(nd));
    nd.px = nb.lo[0]; nd.py = nb.lo[1]; nd.pz = nb.lo[2];
    nd.ex = (uint8_t)e[0]; nd.ey = (uint8_t)e[1]; nd.ez = (uint8_t)e[2];
    nd.child_base = child_base; nd.tri_base = tri_base; nd.magic = KZ_NODE_MAGIC;
    uint32_t triOff = 0, rel = 0; uint8_t imask = 0;
    for (int s = 0; s < 8; ++s) {
        if (childAt[s] < 0) continue;
        const int ci = childAt[s];
        const int c = ch[ci];
        uint8_t *qlo[3] = {nd.qlox, nd.qloy, nd.qloz}, *qhi[3] = {nd.qhix, nd.qhiy, nd.qhiz};
        for (int a = 0; a < 3; ++a) {
            const double sc = ldexp(1.0, e[a] - 127);
            const double lo = floor(((double)bx[ci].lo[a] - (double)nb.lo[a]) / sc);
            const double hi = ceil(((double)bx[ci].hi[a] - (double)nb.lo[a]) / sc);
            qlo[a][s] = (uint8_t)fmin(255.0, fmax(0.0, lo));
            qhi[a][s] = (uint8_t)fmin(255.0, fmax(0.0, hi));
        }
        const uint32_t cnt = sub_count(b, c);
        if (c >= 0 && cnt > KZ_LBVH_MAXLEAF) {
            imask |= (uint8_t)(1u << s);
            WorkItem w; w.bnode = c; w.wnode = child_base + rel;
            cs.out[out_base + rel] = w;
            ++rel;
        } else {
            const uint32_t unary = cnt == 1u ? 1u : (cnt == 2u ? 3u : 7u);
            nd.trimask |= unary << (3 * s);
            const uint32_t first = c < 0 ? (uint32_t)~c : b.first[c];
            for (uint32_t k = 0; k < cnt; ++k) {
                const kzbvh::Tri t = b.tris[ref_tri(b, b.order[first + k])];
                KzF4 *o = cs.tris + 3 * (size_t)(tri_base + triOff + k);
                KzF4 v;
                v.x = t.p[0][0]; v.y = t.p[0][1]; v.z = t.p[0][2]; v.w = __uint_as_float(t.geom); o[0] = v;
                v.x = t.p[1][0]; v.y = t.p[1][1]; v.z = t.p[1][2]; v.w = __uint_as_float(t.prim); o[1] = v;
                v.x = t.p[2][0]; v.y = t.p[2][1]; v.z = t.p[2][2]; v.w = 0.f; o[2] = v;
            }
            triOff += cnt;
        }
    }
    nd.imask = imask;
    cs.nodes[it.wnode] = nd;
    }
}

/* Reference pre-splitting (as in the host SAH builder, kz_bvh_build.h): a triangle whose box is expected to hold other primitives,
 * volume(box) * N / volume(centroid bounds) >= need, gets two references, each bounding the part of the triangle on one side of the
 * spatial median of the box's longest axis.  Clipping is done in float; every reference box is padded by a few ulps of the triangle's
 * largest coordinate and clamped to the triangle's own box, so it contains its part of the triangle and culling stays conservative. */
__global__ void k_make_refs(const kzbvh::Tri *tris, uint32_t n, const uint32_t *bounds, float need, float4 *rlo, float4 *rhi, uint32_t *counter) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const kzbvh::Tri t = tris[i];
    float lo[3], hi[3], ext[3], sext[3], longest = 0.f, mabs = 0.f;
    for (int a = 0; a < 3; ++a) {
        lo[a] = fminf(t.p[0][a], fminf(t.p[1][a], t.p[2][a])); hi[a] = fmaxf(t.p[0][a], fmaxf(t.p[1][a], t.p[2][a]));
        ext[a] = hi[a] - lo[a];
        sext[a] = ord2f(bounds[3 + a]) - ord2f(bounds[a]);
        longest = fmaxf(longest, sext[a]);
        mabs = fmaxf(mabs, fmaxf(fabsf(lo[a]), fabsf(hi[a])));
    }
    double volume = 1.0;
    for (int a = 0; a < 3; ++a) volume *= (double)fmaxf(sext[a], 1e-3f * longest);
    const double inside = volume > 0.0 ? (double)ext[0] * (double)ext[1] * (double)ext[2] * (double)n / volume : 0.0;
    int axis = 0;
    for (int a = 1; a < 3; ++a) if (ext[a] > ext[axis]) axis = a;
    const float plane = 0.5f * (lo[axis] + hi[axis]);
    const bool split = inside >= (double)need && plane > lo[axis] && plane < hi[axis];
    const uint32_t tri_bits = i;
    if (!split) {
        const uint32_t o = atomicAdd(counter, 1u);
        rlo[o] = make_float4(lo[0], lo[1], lo[2], __uint_as_float(tri_bits)); rhi[o] = make_float4(hi[0], hi[1], hi[2], 0.f);
        return;
    }
    float llo[3] = {3.4e38f, 3.4e38f, 3.4e38f}, lhi[3] = {-3.4e38f, -3.4e38f, -3.4e38f};
    float hlo[3] = {3.4e38f, 3.4e38f, 3.4e38f}, hhi[3] = {-3.4e38f, -3.4e38f, -3.4e38f};
    for (int v = 0; v < 3; ++v) {
        const float *a = t.p[v], *b = t.p[(v + 1) % 3];
        if (a[axis] <= plane) for (int k = 0; k < 3; ++k) { llo[k] = fminf(llo[k], a[k]); lhi[k] = fmaxf(lhi[k], a[k]); }
        if (a[axis] >= plane) for (int k = 0; k < 3; ++k) { hlo[k] = fminf(hlo[k], a[k]); hhi[k] = fmaxf(hhi[k], a[k]); }
        if ((a[axis] < plane && b[axis] > plane) || (a[axis] > plane && b[axis] < plane)) {
            const float tt = (plane - a[axis]) / (b[axis] - a[axis]);
            for (int k = 0; k < 3; ++k) {
                const float q = k == axis ? plane : a[k] + tt * (b[k] - a[k]);
                llo[k] = fminf(llo[k], q); lhi[k] = fmaxf(lhi[k], q);
                hlo[k] = fminf(hlo[k], q); hhi[k] = fmaxf(hhi[k], q);
            }
        }
    }
    const float pad = 8.f * 1.1920929e-7f * mabs;
    const uint32_t o = atomicAdd(counter, 2u);
    float4 l, h;
    l = make_float4(fmaxf(llo[0] - pad, lo[0]), fmaxf(llo[1] - pad, lo[1]), fmaxf(llo[2] - pad, lo[2]), __uint_as_float(tri_bits));
    h = make_float4(fminf(lhi[0] + pad, hi[0]), fminf(lhi[1] + pad, hi[1]), fminf(lhi[2] + pad, hi[2]), 0.f);
    rlo[o] = l; rhi[o] = h;
    l = make_float4(fmaxf(hlo[0] - pad, lo[0]), fmaxf(hlo[1] - pad, lo[1]), fmaxf(hlo[2] - pad, lo[2]), __uint_as_float(tri_bits));
    h = make_float4(fminf(hhi[0] + pad, hi[0]), fminf(hhi[1] + pad, hi[1]), fminf(hhi[2] + pad, hi[2]), 0.f);
    rlo[o + 1] = l; rhi[o + 1] = h;
}
#ifndef KZ_LBVH_PRESPLIT_DEFAULT
#define KZ_LBVH_PRESPLIT_DEFAULT 1       /* KZ_LBVH_PRESPLIT=0 turns it off */
#endif

#define KZL_CUDA(call)                                                                                   \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess) {                                                                        \
            err = std::string(#call) + ": " + cudaGetErrorString(e__);                                   \
            for (void *p__ : temp) cudaFreeAsync(p__, s);                                                \
            cudaStreamSynchronize(s);                                                                    \
            return e__ == cudaErrorMemoryAllocation ? KZ_ERR_NOMEM : KZ_ERR_CUDA;                        \
        }                                                                                                \
    } while (0)

#define KZ_LBVH_MAX_LEVELS 31     /* levels the collapse walks; the API accepts KZ_MAX_ACCEL_DEPTH = 30 of them (stack budget in kz_traverse.h) */

/* Builds the accel of the `n_tris_in` device-resident triangles `d_tris` (scene order) on the current device; `r` owns the node and
 * triangle arrays (also after a failure), temporaries are released before returning. */
inline int build(const kzbvh::Tri *d_tris, uint32_t n_tris_in, cudaStream_t s, Result &r, std::string &err) {
    std::vector<void *> temp;
    uint32_t n = n_tris_in;                  /* references: == triangles unless pre-splitting adds some */
    r = Result();
    if (n == 0) return KZ_OK;
    /* temporaries come from the device's stream-ordered pool: with peer access enabled (multi-device contexts, NCCL) every plain
     * cudaMalloc maps the new block into all peers, which made this build 12x slower on two GPUs than on one */
    auto talloc = [&](size_t bytes, void **p) { cudaError_t e = cudaMallocAsync(p, std::max<size_t>(bytes, 16), s); if (e == cudaSuccess) temp.push_back(*p); return e; };
    unsigned long long *k0, *k1; uint32_t *v0, *v1, *bounds;
    KZL_CUDA(talloc(64, (void **)&bounds));
    const uint32_t init[8] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0u, 0u, 0u, 0u, 0u};
    KZL_CUDA(cudaMemcpyAsync(bounds, init, sizeof(init), cudaMemcpyHostToDevice, s));
    k_scene_bounds<<<std::min((n + 255u) / 256u, 148u * 8u), 256, 0, s>>>(d_tris, n, bounds);
    ++r.launches;
    float4 *rlo = nullptr, *rhi = nullptr;
    {
        const char *e = getenv("KZ_LBVH_PRESPLIT");
        const bool presplit = e ? atoi(e) != 0 : KZ_LBVH_PRESPLIT_DEFAULT != 0;
        if (presplit && n_tris_in >= 64u && n_tris_in < 0x3FFFFFFFu) {
            const char *ne = getenv("KZ_SAH_PRESPLIT_NEED");
            const float need = ne ? (float)atof(ne) : 0.25f;
            KZL_CUDA(talloc((size_t)n * 2 * sizeof(float4), (void **)&rlo)); KZL_CUDA(talloc((size_t)n * 2 * sizeof(float4), (void **)&rhi));
            KZL_CUDA(cudaMemsetAsync(bounds + 8, 0, 4, s));
            k_make_refs<<<(n + 255u) / 256u, 256, 0, s>>>(d_tris, n, bounds, need, rlo, rhi, bounds + 8);
            ++r.launches;
            uint32_t nref = 0;
            KZL_CUDA(cudaMemcpyAsync(&nref, bounds + 8, 4, cudaMemcpyDeviceToHost, s));
            KZL_CUDA(cudaStreamSynchronize(s));
            /* kept only when at least a quarter of the triangles qualified: a soup (86 % on the 2^20-triangle one: +5-7 % rays/s) profits,
             * a surface mesh with a few outsized triangles does not (the host builder's cost arbitration drops those trees, item 22) */
            if ((unsigned long long)(nref - n_tris_in) * 4ull >= (unsigned long long)n_tris_in) n = nref;
            else { rlo = nullptr; rhi = nullptr; }
        }
    }
    KZL_CUDA(talloc((size_t)n * 8, (void **)&k0)); KZL_CUDA(talloc((size_t)n * 8, (void **)&k1));
    KZL_CUDA(talloc((size_t)n * 4, (void **)&v0)); KZL_CUDA(talloc((size_t)n * 4, (void **)&v1));
    const unsigned blocks = (n + 255u) / 256u;
    k_morton<<<blocks, 256, 0, s>>>(d_tris, rlo, rhi, n, bounds, k0, v0);
    ++r.launches;
    cub::DoubleBuffer<unsigned long long> dk(k0, k1);
    cub::DoubleBuffer<uint32_t> dv(v0, v1);
    size_t sort_bytes = 0;
    KZL_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, dk, dv, (int)n, 0, 63, s));
    void *sort_tmp;
    KZL_CUDA(talloc(sort_bytes, &sort_tmp));
    KZL_CUDA(cub::DeviceRadixSort::SortPairs(sort_tmp, sort_bytes, dk, dv, (int)n, 0, 63, s));
    r.launches += 8;

    BuildState b;
    b.tris = d_tris; b.rlo = rlo; b.rhi = rhi; b.n = n; b.order = dv.Current(); b.keys = dk.Current();
    const size_t ni = n > 1 ? n - 1 : 1;
    KZL_CUDA(talloc(ni * 4, (void **)&b.left)); KZL_CUDA(talloc(ni * 4, (void **)&b.right));
    KZL_CUDA(talloc((size_t)(2 * (size_t)n) * 4, (void **)&b.parent));
    KZL_CUDA(talloc(ni * 4, (void **)&b.first)); KZL_CUDA(talloc(ni * 4, (void **)&b.last));
    KZL_CUDA(talloc(ni * 16, (void **)&b.blo)); KZL_CUDA(talloc(ni * 16, (void **)&b.bhi));
    KZL_CUDA(talloc(ni * 4, (void **)&b.flags));
    KZL_CUDA(cudaMemsetAsync(b.flags, 0, ni * 4, s));
    if (n > 1) {
        k_karras<<<(n - 1 + 255u) / 256u, 256, 0, s>>>(b);
        k_fit<<<blocks, 256, 0, s>>>(b);
        r.launches += 2;
    }
    /* output arrays: every wide node except the root has >= 2 children below it... an upper bound
     * of n nodes is loose but safe (a wide node owns >= 1 triangle or >= 2 wide children) */
    KzNode8 *d_nodes; KzF4 *d_out_tris; uint32_t *counters; WorkItem *w0, *w1;
    const size_t max_nodes = (size_t)n;
    KZL_CUDA(r.nodes.alloc(max_nodes * sizeof(KzNode8))); d_nodes = r.nodes.as<KzNode8>();
    KZL_CUDA(r.tris.alloc((size_t)n * 3 * sizeof(KzF4))); d_out_tris = r.tris.as<KzF4>();
    /* counters[0] = wide nodes (root taken), [1] = emitted triangles, [2 + l] = work items of level l */
    uint32_t cinit[4 + KZ_LBVH_MAX_LEVELS];
    memset(cinit, 0, sizeof(cinit));
    cinit[0] = 1u; cinit[2] = 1u;
    KZL_CUDA(talloc(sizeof(cinit), (void **)&counters));
    KZL_CUDA(talloc(max_nodes * sizeof(WorkItem), (void **)&w0)); KZL_CUDA(talloc(max_nodes * sizeof(WorkItem), (void **)&w1));
    KZL_CUDA(cudaMemcpyAsync(counters, cinit, sizeof(cinit), cudaMemcpyHostToDevice, s));
    WorkItem rootItem; rootItem.bnode = n > 1 ? 0 : ~0; rootItem.wnode = 0;
    KZL_CUDA(cudaMemcpyAsync(w0, &rootItem, sizeof(rootItem), cudaMemcpyHostToDevice, s));
    CollapseState cs;
    cs.b = b; cs.nodes = d_nodes; cs.tris = d_out_tris; cs.node_counter = counters; cs.tri_counter = counters + 1;
    /* level-synchronous, but without a host round trip per level: every launch reads its item count from HBM; the grid is sized
     * for the widest possible level of its depth (8^l items) and capped at a few waves, with a grid-stride loop inside */
    int dev = 0, sms = 148;
    cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    WorkItem *in = w0, *out = w1;
    double widest = 1.0;
    for (int l = 0; l < KZ_LBVH_MAX_LEVELS; ++l) {
        cs.in = in; cs.out = out; cs.in_count = counters + 2 + l; cs.out_count = counters + 3 + l;
        const double cap = std::min(widest, (double)max_nodes);
        const unsigned grid = (unsigned)std::min<double>((cap + 63.0) / 64.0, (double)sms * 32.0);
        k_collapse<<<std::max(1u, grid), 64, 0, s>>>(cs);
        ++r.launches;
        widest *= 8.0;
        std::swap(in, out);
    }
    uint32_t fin[3 + KZ_LBVH_MAX_LEVELS]; uint32_t hb[8];
    KZL_CUDA(cudaMemcpyAsync(fin, counters, sizeof(fin), cudaMemcpyDeviceToHost, s));
    KZL_CUDA(cudaMemcpyAsync(hb, bounds, 32, cudaMemcpyDeviceToHost, s));
    KZL_CUDA(cudaStreamSynchronize(s));
    KZL_CUDA(cudaGetLastError());
    r.n_nodes = fin[0]; r.n_tris = fin[1];
    r.max_abs = ord2f(hb[6]);
    for (int l = 0; l < KZ_LBVH_MAX_LEVELS && fin[2 + l] != 0u; ++l) r.depth = l + 1;
    /* level l + 1 is allocated (node_counter) while level l runs, so the levels are consecutive ranges in launch order */
    r.level_first.assign(1, 0u);
    for (int l = 0; l < r.depth; ++l) r.level_first.push_back(r.level_first.back() + fin[2 + l]);
    for (void *p : temp) cudaFreeAsync(p, s);
    cudaStreamSynchronize(s);
    if (fin[2 + KZ_LBVH_MAX_LEVELS] != 0u) { err = "lbvh: accel deeper than the traversal stack allows"; return KZ_ERR_UNSUPPORTED; }
    if (r.n_tris != n) { err = "lbvh: triangle count mismatch after collapse"; return KZ_ERR_CUDA; }
    return KZ_OK;
}

}  // namespace kzlbvh
#endif
