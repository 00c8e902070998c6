/* kz_traverse.h -- closest-hit traversal of the 8-wide compressed BVH + the parity-contracted
 * triangle test.  Replaces rtcIntersect1 as called at src/kazen/accel.cpp:98.
 *
 * Triangle test: Embree's robust ("Pluecker") single-ray test on origin-relative vertices with
 * the operation shapes of its AVX2 build (fused dot/cross); every operation is an explicitly
 * rounded intrinsic so nvcc cannot re-associate or contract differently from the oracle
 * (oracle/kzo_accel.h): hit IDs and t are bit-identical to the oracle by construction, as long
 * as culling is conservative.
 *
 * Culling is conservative by construction:
 *   - child boxes are quantised outwards (lo rounded down, hi rounded up) at build time;
 *   - every ray widens each slab by `slack` = 2^-18 * (max|org| + scene_max_abs) in position
 *     space by shifting the origin used for the near / far plane (no per-child cost); this
 *     covers the Pluecker tolerance (FLT_EPSILON*|UVW|), the rounding of p - org, and the
 *     rounding of the slab FMAs, all of which are a few ulp of those magnitudes;
 *   - |dir| components below 1e-18 are replaced by +-1e-18 (Embree's rcp_safe idea), so the
 *     slab arithmetic never produces NaN.
 *   Ties on exact t are broken by smallest (geomID, primID), independent of traversal order.
 *
 * Traversal: stack of (node group | triangle group) 8-byte entries, octant-ordered child
 * visiting (slot ^ ray octant, no distance sort), short stack in shared memory on the device
 * with overflow to local memory.  The 8 slab tests of a node step leave one sign bit each in a
 * byte (slot order); the inner-child hits are that byte & imask with its bits permuted by the ray
 * octant (three masked swaps), the leaf hits are the byte spread to 3 bits per slot & trimask:
 * word-parallel, no per-child shifts (the node step is bound by instruction issue and by the
 * ALU pipe: 281 -> ~240 instructions, 128 -> ~85 of them on the ALU pipe).
 */
#ifndef KZ_TRAVERSE_H
#define KZ_TRAVERSE_H
#include "kz_scene.h"

struct KzHit { float t, u, v; uint32_t prim, geom; };

#if KZ_DEVICE_CODE
#define KZ_LDG_U4(ptr) __ldg(reinterpret_cast<const uint4 *>(ptr))
KZ_HD KzU4 kz_load_u4(const void *p) { uint4 v = KZ_LDG_U4(p); KzU4 r; r.x = v.x; r.y = v.y; r.z = v.z; r.w = v.w; return r; }
#else
KZ_HD KzU4 kz_load_u4(const void *p) { KzU4 r; memcpy(&r, p, 16); return r; }
#endif

KZ_HD float kz_edot(float ax, float ay, float az, float bx, float by, float bz) {
    return kz_fma(ax, bx, kz_fma(ay, by, kz_mul(az, bz)));
}
/* a*b - c fused */
KZ_HD float kz_fms(float a, float b, float c) { return kz_fma(a, b, -c); }

/* Returns true if the triangle is hit inside [tnear, tfar]; fills t,u,v. */
KZ_HD bool kz_pluecker(float ox, float oy, float oz, float dx, float dy, float dz, float tnear, float tfar,
                       KzU4 a, KzU4 b, KzU4 c, float &t_out, float &u_out, float &v_out) {
    float v0x = kz_sub(kz_u2f(a.x), ox), v0y = kz_sub(kz_u2f(a.y), oy), v0z = kz_sub(kz_u2f(a.z), oz);
    float v1x = kz_sub(kz_u2f(b.x), ox), v1y = kz_sub(kz_u2f(b.y), oy), v1z = kz_sub(kz_u2f(b.z), oz);
    float v2x = kz_sub(kz_u2f(c.x), ox), v2y = kz_sub(kz_u2f(c.y), oy), v2z = kz_sub(kz_u2f(c.z), oz);
    float e0x = kz_sub(v2x, v0x), e0y = kz_sub(v2y, v0y), e0z = kz_sub(v2z, v0z);
    float e1x = kz_sub(v0x, v1x), e1y = kz_sub(v0y, v1y), e1z = kz_sub(v0z, v1z);
    float e2x = kz_sub(v1x, v2x), e2y = kz_sub(v1y, v2y), e2z = kz_sub(v1z, v2z);
    /* U = dot(cross(e0, v2+v0), D) etc. */
    float s0x = kz_add(v2x, v0x), s0y = kz_add(v2y, v0y), s0z = kz_add(v2z, v0z);
    float s1x = kz_add(v0x, v1x), s1y = kz_add(v0y, v1y), s1z = kz_add(v0z, v1z);
    float s2x = kz_add(v1x, v2x), s2y = kz_add(v1y, v2y), s2z = kz_add(v1z, v2z);
    float U = kz_edot(kz_fms(e0y, s0z, kz_mul(e0z, s0y)), kz_fms(e0z, s0x, kz_mul(e0x, s0z)), kz_fms(e0x, s0y, kz_mul(e0y, s0x)), dx, dy, dz);
    float V = kz_edot(kz_fms(e1y, s1z, kz_mul(e1z, s1y)), kz_fms(e1z, s1x, kz_mul(e1x, s1z)), kz_fms(e1x, s1y, kz_mul(e1y, s1x)), dx, dy, dz);
    float W = kz_edot(kz_fms(e2y, s2z, kz_mul(e2z, s2y)), kz_fms(e2z, s2x, kz_mul(e2x, s2z)), kz_fms(e2x, s2y, kz_mul(e2y, s2x)), dx, dy, dz);
    float UVW = kz_add(kz_add(U, V), W);
    float eps = kz_mul(1.1920928955078125e-07f, fabsf(UVW));
    float mn = fminf(U, fminf(V, W)), mx = fmaxf(U, fmaxf(V, W));
    if (!(mn >= -eps || mx <= eps)) return false;
    /* stable_triangle_normal(e0, e1, e2) */
    float ab_x = kz_mul(e0z, e1y), ab_y = kz_mul(e0x, e1z), ab_z = kz_mul(e0y, e1x);
    float bc_x = kz_mul(e1z, e2y), bc_y = kz_mul(e1x, e2z), bc_z = kz_mul(e1y, e2x);
    float cab_x = kz_fms(e0y, e1z, ab_x), cab_y = kz_fms(e0z, e1x, ab_y), cab_z = kz_fms(e0x, e1y, ab_z);
    float cbc_x = kz_fms(e1y, e2z, bc_x), cbc_y = kz_fms(e1z, e2x, bc_y), cbc_z = kz_fms(e1x, e2y, bc_z);
    float ngx = fabsf(ab_x) < fabsf(bc_x) ? cab_x : cbc_x;
    float ngy = fabsf(ab_y) < fabsf(bc_y) ? cab_y : cbc_y;
    float ngz = fabsf(ab_z) < fabsf(bc_z) ? cab_z : cbc_z;
    float d = kz_edot(ngx, ngy, ngz, dx, dy, dz);
    float den = kz_add(d, d);
    float T0 = kz_edot(v0x, v0y, v0z, ngx, ngy, ngz);
    float T = kz_add(T0, T0);
    float t = kz_mul(kz_rcp(den), T);
    if (!(tnear <= t && t <= tfar)) return false;
    if (den == 0.0f) return false;
    float rcpUVW = fabsf(UVW) < 1e-18f ? 0.0f : kz_rcp(UVW);
    t_out = t;
    u_out = fminf(kz_mul(U, rcpUVW), 1.0f);
    v_out = fminf(kz_mul(V, rcpUVW), 1.0f);
    return true;
}

KZ_HD float kz_magic_adjust(float v, float k) { return fmaf(fabsf(v), k, v); }
KZ_HD float kz_rcp_safe(float d) {
    if (fabsf(d) < 1e-18f) d = (kz_f2u(d) >> 31) ? -1e-18f : 1e-18f;
#if KZ_DEVICE_CODE
    /* culling only: the approximate reciprocal (one MUFU instead of the IEEE division's ~8 instructions, three per ray) is within 2 ulp,
     * i.e. 2^-22 |p - o| in position space, far inside the slack */
    float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d)); return r;
#else
    return 1.0f / d;
#endif
}

#ifndef KZ_PRMT_AXES
#define KZ_PRMT_AXES 36     /* bit mask: near x,y,z = 1,2,4; far x,y,z = 8,16,32.  Measured (Mrays/s primary / incoherent, 2^20-triangle soup):
                             * 0 -> 2572 / 2029, 7 -> 2862 / 2082, 15 -> 2810 / 2077, 31 -> 2779 / 2071, 36 -> 2902 / 2103: 16 of the 48
                             * conversions on the ALU pipe (rate 1/2), 32 on the XU pipe (rate 1/4) balance the two */
#endif
#ifndef KZ_SLACK
#define KZ_SLACK 3.814697265625e-06f
#endif
#ifndef KZ_SHORT_STACK
#define KZ_SHORT_STACK 8          /* entries per thread kept in shared memory */
#endif
#define KZ_LOCAL_STACK (64 - KZ_SHORT_STACK)   /* overflow entries in local memory */
/* Stack budget (64 entries): a node step leaves at most one entry (the siblings of the child it descends into), i.e. at most
 * `depth` entries at any time; a postponed triangle group takes two and is only put aside while fewer than
 * KZ_POSTPONE_SP_LIMIT entries are stacked.  32 + 2 + KZ_MAX_ACCEL_DEPTH = 64. */
#define KZ_POSTPONE_SP_LIMIT 32
#define KZ_MAX_ACCEL_DEPTH (KZ_SHORT_STACK + KZ_LOCAL_STACK - 2 - KZ_POSTPONE_SP_LIMIT)

#ifndef KZ_TRACE_THREADS
#define KZ_TRACE_THREADS 128      /* threads per CTA of every kernel that traverses (kz_kernels.cuh) */
#endif
struct KzStackRef {
#if defined(__CUDACC__)
    uint32_t sbase;               /* shared-window byte address of this thread's column: entry i at sbase + i * 8 * KZ_TRACE_THREADS */
    uint32_t lbase;               /* shared-window byte address of the look-up tables: 8 x 256 bytes (octant permutation), 256 words (spread) */
#endif
};

/* Look-up tables of the node step (2 KB + 1 KB): the octant permutation of an 8-bit child mask (bit j -> bit j ^ c) and the
 * spread of 8 child bits to 3 bits per slot.  On the device they sit in shared memory (filled by kz_trav_shared_init at the top of
 * every traversing kernel): two loads replace ~25 bit operations of the issue-bound node step. */
KZ_HD uint32_t kz_perm8(uint32_t m, uint32_t c) {
    if (c & 1u) m = ((m & 0x55u) << 1) | ((m >> 1) & 0x55u);
    if (c & 2u) m = ((m & 0x33u) << 2) | ((m >> 2) & 0x33u);
    if (c & 4u) m = ((m & 0x0Fu) << 4) | (m >> 4);
    return m;
}
KZ_HD uint32_t kz_spread7(uint32_t m) {
    m = (m | (m << 8)) & 0x0000F00Fu;
    m = (m | (m << 4)) & 0x000C30C3u;
    m = (m | (m << 2)) & 0x00249249u;
    return m * 7u;
}
#if defined(__CUDACC__)
__shared__ uint32_t kz_s_lut[512 + 256];      /* [0, 2048) bytes: perm8 by octant; then 256 words: spread7 */
__shared__ uint2    kz_s_stack[KZ_SHORT_STACK * KZ_TRACE_THREADS];
__device__ __forceinline__ KzStackRef kz_trav_shared_init() {
    uint8_t *perm = reinterpret_cast<uint8_t *>(kz_s_lut);
    for (uint32_t i = threadIdx.x; i < 8u * 256u; i += blockDim.x) perm[i] = (uint8_t)kz_perm8(i & 255u, i >> 8);
    for (uint32_t i = threadIdx.x; i < 256u; i += blockDim.x) kz_s_lut[512 + i] = kz_spread7(i);
    __syncthreads();
    /* both addresses go through a volatile asm so that they stay in registers: left alone, the compiler recomputes the CTA's
     * shared-window base (S2UR CgaCtaId, UMOV, ULEA ...) at every push, pop and table look-up of the node step */
    KzStackRef stk;
    stk.sbase = (uint32_t)__cvta_generic_to_shared(kz_s_stack + threadIdx.x);
    stk.lbase = (uint32_t)__cvta_generic_to_shared(kz_s_lut);
    asm volatile("mov.b32 %0, %0;" : "+r"(stk.sbase));
    asm volatile("mov.b32 %0, %0;" : "+r"(stk.lbase));
    return stk;
}
__device__ __forceinline__ uint32_t kz_lds_u8(uint32_t a) { uint32_t r; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(r) : "r"(a)); return r; }
__device__ __forceinline__ uint32_t kz_lds_u32(uint32_t a) { uint32_t r; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r) : "r"(a)); return r; }
#endif

/* Per-ray traversal state.  The loop is split into steps (init / node / triangle / pop) so that the
 * same arithmetic serves the plain per-ray loop below (kz_trace: host emulation, BSDF-side helpers)
 * and the warp-cooperative persistent loop of kz_kernels.cuh (lane refill + postponed leaf tests). */
struct KzTrav {
    float ox, oy, oz, dx, dy, dz, tmin;
    float rdx, rdy, rdz;
    float cnx, cny, cnz, cfx, cfy, cfz;      /* -(o' * rd) for the near / far planes, o' = origin moved by the slack (widened slab) */
    uint32_t oct_inv;                        /* 7 - ray octant */
    KzHit best;
    uint32_t ng_x, ng_y;                     /* node group: (child base, hits<<24 | imask) */
    uint32_t tg_x, tg_y, tg_m;               /* triangle group: (tri base, hit bits in trimask positions, trimask) */
    int sp;                                  /* stacked entries */
};
struct KzLocalStack { uint32_t x[KZ_LOCAL_STACK], y[KZ_LOCAL_STACK]; };

/* False if a traversal of this ray is an immediate miss: an empty accel, or a NaN component (see kz_trav_init). */
KZ_HD bool kz_trav_starts(const KzScene &sc, float ox, float oy, float oz, float dx, float dy, float dz, float tmin, float tmax) {
    const bool has_nan = isnan(ox) || isnan(oy) || isnan(oz) || isnan(dx) || isnan(dy) || isnan(dz) || isnan(tmin) || isnan(tmax);
    return sc.n_nodes != 0 && !has_nan;
}

KZ_HD void kz_trav_init(const KzScene &sc, KzTrav &t, float ox, float oy, float oz, float dx, float dy, float dz, float tmin, float tmax) {
    t.ox = ox; t.oy = oy; t.oz = oz; t.dx = dx; t.dy = dy; t.dz = dz; t.tmin = tmin;
    t.best.t = tmax; t.best.u = 0.f; t.best.v = 0.f; t.best.prim = KZ_INVALID_ID; t.best.geom = KZ_INVALID_ID;
    const float slack = (fmaxf(fabsf(ox), fmaxf(fabsf(oy), fabsf(oz))) + sc.scene_max_abs) * KZ_SLACK;
    t.rdx = kz_rcp_safe(dx); t.rdy = kz_rcp_safe(dy); t.rdz = kz_rcp_safe(dz);
    const bool nx = t.rdx < 0.f, ny = t.rdy < 0.f, nz = t.rdz < 0.f;
    /* plane distances are p * rd - o' * rd (one FMA per axis and side in the node step); the rounding of o' * rd is 2^-24 |o'| in
     * position space, 1/64 of the slack */
    t.cnx = -((nx ? ox - slack : ox + slack) * t.rdx); t.cfx = -((nx ? ox + slack : ox - slack) * t.rdx);
    t.cny = -((ny ? oy - slack : oy + slack) * t.rdy); t.cfy = -((ny ? oy + slack : oy - slack) * t.rdy);
    t.cnz = -((nz ? oz - slack : oz + slack) * t.rdz); t.cfz = -((nz ? oz + slack : oz - slack) * t.rdz);
    t.oct_inv = ((nx ? 0u : 1u) | (ny ? 0u : 2u) | (nz ? 0u : 4u));
    /* A ray with a NaN component can never be accepted by the triangle test (every comparison fails), but fminf/fmaxf drop
     * NaNs, so the slab test would let it walk the whole tree.  Such rays do occur -- the reference's cosine-hemisphere warp
     * yields sqrt(-eps) for a sample that is exactly 0 (warp.cpp:85-115) -- so they are turned into an immediate miss. */
    t.ng_x = 0u; t.ng_y = kz_trav_starts(sc, ox, oy, oz, dx, dy, dz, tmin, tmax) ? 0x80000000u : 0u;      /* root, or nothing to do */
    t.tg_x = 0u; t.tg_y = 0u; t.tg_m = 0u;
    t.sp = 0;
}

KZ_HD void kz_trav_push(KzTrav &t, const KzStackRef &stk, KzLocalStack &ls, uint32_t x, uint32_t y) {
#if KZ_DEVICE_CODE
    if (t.sp < KZ_SHORT_STACK) asm volatile("st.shared.v2.u32 [%0], {%1, %2};" :: "r"(stk.sbase + (uint32_t)t.sp * (8u * KZ_TRACE_THREADS)), "r"(x), "r"(y) : "memory");
    else { ls.x[t.sp - KZ_SHORT_STACK] = x; ls.y[t.sp - KZ_SHORT_STACK] = y; }
#else
    (void)stk; ls.x[t.sp] = x; ls.y[t.sp] = y;
#endif
    ++t.sp;
}
KZ_HD void kz_trav_pop1(KzTrav &t, const KzStackRef &stk, const KzLocalStack &ls, uint32_t &x, uint32_t &y) {
    --t.sp;
#if KZ_DEVICE_CODE
    if (t.sp < KZ_SHORT_STACK) asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(x), "=r"(y) : "r"(stk.sbase + (uint32_t)t.sp * (8u * KZ_TRACE_THREADS)) : "memory");
    else { x = ls.x[t.sp - KZ_SHORT_STACK]; y = ls.y[t.sp - KZ_SHORT_STACK]; }
#else
    (void)stk; x = ls.x[t.sp]; y = ls.y[t.sp];
#endif
}
/* Pops the next piece of work: a node group goes to ng; a postponed triangle group (y <= 0x00FFFFFF, two entries: see
 * kz_trav_postpone) goes to tg and leaves ng empty. */
KZ_HD void kz_trav_pop(KzTrav &t, const KzStackRef &stk, const KzLocalStack &ls) {
    kz_trav_pop1(t, stk, ls, t.ng_x, t.ng_y);
    if (t.ng_y <= 0x00FFFFFFu) {
        uint32_t unused;
        t.tg_x = t.ng_x; t.tg_y = t.ng_y; t.ng_x = 0u; t.ng_y = 0u;
        kz_trav_pop1(t, stk, ls, t.tg_m, unused);
    }
}
/* Puts the rest of the current triangle group aside (the warp-cooperative loop does that while too few lanes hold triangles). */
KZ_HD void kz_trav_postpone(KzTrav &t, const KzStackRef &stk, KzLocalStack &ls) {
    kz_trav_push(t, stk, ls, t.tg_m, 0u);
    kz_trav_push(t, stk, ls, t.tg_x, t.tg_y);
    t.tg_y = 0u;
}

/* Takes the next child of the current node group (ng_y > 0x00FFFFFF), intersects its 8 child boxes and
 * leaves the new node group in ng and the new triangle group in tg. */
KZ_HD void kz_trav_node(const KzScene &sc, KzTrav &t, const KzStackRef &stk, KzLocalStack &ls) {
    const uint32_t hits_imask = t.ng_y;
    const uint32_t bit = kz_bfind(hits_imask);
    const uint32_t child_base = t.ng_x;
    t.ng_y &= ~(1u << bit);
    if (t.ng_y > 0x00FFFFFFu) kz_trav_push(t, stk, ls, t.ng_x, t.ng_y);     /* siblings left: push the rest of the group */
    const uint32_t slot = (bit - 24u) ^ t.oct_inv;
    const uint32_t rel = kz_popc(hits_imask & ~(0xFFFFFFFFu << slot));
    const KzNode8 *node = sc.nodes + (child_base + rel);
    const KzU4 n0 = kz_load_u4(reinterpret_cast<const char *>(node));
    const KzU4 n1 = kz_load_u4(reinterpret_cast<const char *>(node) + 16);
    const KzU4 n2 = kz_load_u4(reinterpret_cast<const char *>(node) + 32);
    const KzU4 n3 = kz_load_u4(reinterpret_cast<const char *>(node) + 48);
    const KzU4 n4 = kz_load_u4(reinterpret_cast<const char *>(node) + 64);
    const float px = kz_u2f(n0.x), py = kz_u2f(n0.y), pz = kz_u2f(n0.z);
    const uint32_t ex = n0.w & 0xFFu, ey = (n0.w >> 8) & 0xFFu, ez = (n0.w >> 16) & 0xFFu, imask = n0.w >> 24;
    /* t = q * (2^e * rd) + (p * rd - o' * rd) */
    const float adx = kz_u2f(ex << 23) * t.rdx, ady = kz_u2f(ey << 23) * t.rdy, adz = kz_u2f(ez << 23) * t.rdz;
    const float anx = fmaf(px, t.rdx, t.cnx), any_ = fmaf(py, t.rdy, t.cny), anz = fmaf(pz, t.rdz, t.cnz);
    const float afx = fmaf(px, t.rdx, t.cfx), afy = fmaf(py, t.rdy, t.cfy), afz = fmaf(pz, t.rdz, t.cfz);
    /* plane constants for the permute-built operands (32768 + q): a - 32768*ad, moved outwards by 2^-22 |.| which covers the
     * rounding of this extra operation (<= 2^-24 |.|), so culling stays conservative */
#define KZ_MAGIC_NEAR(a, ad) kz_magic_adjust(fmaf(-32768.f, ad, a), -2.384185791015625e-07f)
#define KZ_MAGIC_FAR(a, ad) kz_magic_adjust(fmaf(-32768.f, ad, a), 2.384185791015625e-07f)
    const float anx_m = KZ_MAGIC_NEAR(anx, adx), any_m = KZ_MAGIC_NEAR(any_, ady), anz_m = KZ_MAGIC_NEAR(anz, adz);
    const float afx_m = KZ_MAGIC_FAR(afx, adx), afy_m = KZ_MAGIC_FAR(afy, ady), afz_m = KZ_MAGIC_FAR(afz, adz);
#undef KZ_MAGIC_NEAR
#undef KZ_MAGIC_FAR
    const bool nx = !(t.oct_inv & 1u), ny = !(t.oct_inv & 2u), nz = !(t.oct_inv & 4u);
    /* one bit per child, slot 7 first so that slot j ends up at bit j: the sign of cmax - cmin (set = missed).  The operands are
     * never NaN (kz_trav_init), an infinite cmin or cmax keeps the sign right, and inf - inf = +NaN reads as a hit (conservative). */
    uint32_t miss = 0u;
    /* the permute takes ONE immediate operand, which should be the selector: its other input, the word 0x47000000, therefore
     * comes out of the node (KzNode8::magic) -- as a literal the compiler puts IT into the immediate slot and moves every
     * selector into a register first (13 instructions for 8 permutes) */
    const uint32_t magic = n1.w;
#if KZ_DEVICE_CODE
#pragma unroll
#endif
    for (int half = 1; half >= 0; --half) {
        const uint32_t qlox = half ? n2.y : n2.x, qloy = half ? n2.w : n2.z, qloz = half ? n3.y : n3.x;
        const uint32_t qhix = half ? n3.w : n3.z, qhiy = half ? n4.y : n4.x, qhiz = half ? n4.w : n4.z;
        const uint32_t qnx = nx ? qhix : qlox, qfx = nx ? qlox : qhix;
        const uint32_t qny = ny ? qhiy : qloy, qfy = ny ? qloy : qhiy;
        const uint32_t qnz = nz ? qhiz : qloz, qfz = nz ? qloz : qhiz;
        /* byte -> float: either a conversion (I2F.U8, XU pipe) or the bit pattern 0x4700bb00 = 32768 + b built by one
         * byte permute (ALU pipe) with the 32768 folded into the plane constant; KZ_PRMT_AXES spreads the 48 conversions
         * of a node step over the two pipes. */
#define KZ_Q2F(w, J) ((float)(((w) >> (8 * (J))) & 0xFFu))
#define KZ_Q2M(w, J) kz_u2f(kz_byte_perm_sel((w), magic, 0x7404 | ((J) << 4)))
#define KZ_CHILD(J) { \
            const float tnx = (KZ_PRMT_AXES & 1) ? fmaf(KZ_Q2M(qnx, J), adx, anx_m) : fmaf(KZ_Q2F(qnx, J), adx, anx); \
            const float tny = (KZ_PRMT_AXES & 2) ? fmaf(KZ_Q2M(qny, J), ady, any_m) : fmaf(KZ_Q2F(qny, J), ady, any_); \
            const float tnz = (KZ_PRMT_AXES & 4) ? fmaf(KZ_Q2M(qnz, J), adz, anz_m) : fmaf(KZ_Q2F(qnz, J), adz, anz); \
            const float tfx = (KZ_PRMT_AXES & 8) ? fmaf(KZ_Q2M(qfx, J), adx, afx_m) : fmaf(KZ_Q2F(qfx, J), adx, afx); \
            const float tfy = (KZ_PRMT_AXES & 16) ? fmaf(KZ_Q2M(qfy, J), ady, afy_m) : fmaf(KZ_Q2F(qfy, J), ady, afy); \
            const float tfz = (KZ_PRMT_AXES & 32) ? fmaf(KZ_Q2M(qfz, J), adz, afz_m) : fmaf(KZ_Q2F(qfz, J), adz, afz); \
            const float cmin = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, t.tmin)); \
            const float cmax = fminf(fminf(tfx, tfy), fminf(tfz, t.best.t)); \
            miss = kz_shl1_sign(miss, cmax - cmin); }
        KZ_CHILD(3) KZ_CHILD(2) KZ_CHILD(1) KZ_CHILD(0)
#undef KZ_CHILD
#undef KZ_Q2F
#undef KZ_Q2M
    }
    const uint32_t hit8 = ~miss & 0xFFu;
    /* inner children: visiting order is slot ^ octant, highest first (kz_bfind): bit j moves to j ^ oct_inv;
     * leaf children: bit j -> bits 3j..3j+2, masked by the triangles the slot really has */
#if KZ_DEVICE_CODE
    const uint32_t hi = kz_lds_u8(stk.lbase + (t.oct_inv << 8) + (hit8 & imask));
    const uint32_t sp7 = kz_lds_u32(stk.lbase + 2048u + (hit8 << 2));
#else
    const uint32_t hi = kz_perm8(hit8 & imask, t.oct_inv);
    const uint32_t sp7 = kz_spread7(hit8);
#endif
    t.ng_x = n1.x;
    t.ng_y = (hi << 24) | imask;
    t.tg_x = n1.y;
    t.tg_m = n1.z;
    t.tg_y = sp7 & n1.z;
}

/* True if the ray cannot touch the box [lo, hi] before `tfar`: the slab test of the node step (same widened origin), on exact bounds. */
KZ_HD bool kz_trav_misses_box(const KzTrav &t, const float *lo, const float *hi, float tfar) {
    const bool nx = !(t.oct_inv & 1u), ny = !(t.oct_inv & 2u), nz = !(t.oct_inv & 4u);
    const float tnx = fmaf(nx ? hi[0] : lo[0], t.rdx, t.cnx), tfx = fmaf(nx ? lo[0] : hi[0], t.rdx, t.cfx);
    const float tny = fmaf(ny ? hi[1] : lo[1], t.rdy, t.cny), tfy = fmaf(ny ? lo[1] : hi[1], t.rdy, t.cfy);
    const float tnz = fmaf(nz ? hi[2] : lo[2], t.rdz, t.cnz), tfz = fmaf(nz ? lo[2] : hi[2], t.rdz, t.cfz);
    const float cmin = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, t.tmin));
    const float cmax = fminf(fminf(tfx, tfy), fminf(tfz, tfar));
    return cmin > cmax;          /* a NaN says "may touch" */
}

/* Tests the next triangle of the current triangle group (tg_y != 0); returns true if it became the best hit. */
KZ_HD bool kz_trav_tri(const KzScene &sc, KzTrav &t) {
    const uint32_t ti = kz_bfind(t.tg_y);
    t.tg_y &= ~(1u << ti);
    const KzF4 *tp = sc.tris + (size_t)(t.tg_x + kz_popc(t.tg_m & ~(0xFFFFFFFFu << ti))) * 3;
    const KzU4 a = kz_load_u4(tp), b = kz_load_u4(tp + 1), c = kz_load_u4(tp + 2);
    float tt, u, v;
    if (kz_pluecker(t.ox, t.oy, t.oz, t.dx, t.dy, t.dz, t.tmin, t.best.t, a, b, c, tt, u, v)) {
        const uint32_t geom = a.w, prim = b.w;
        const bool better = tt < t.best.t || geom < t.best.geom || (geom == t.best.geom && prim < t.best.prim);
        if (better) { t.best.t = tt; t.best.u = u; t.best.v = v; t.best.geom = geom; t.best.prim = prim; }
        return better;
    }
    return false;
}

/* The seed test: true if the ray (o, d) hits triangle `prim` of mesh `geom` (a hint, e.g. what this ray's pixel hit last time) inside
 * [tmin, tmax]; fills `h` with that hit.  An index out of range, or KZ_INVALID_ID, is no hit, and so is every ray whose traversal would be
 * an immediate miss (kz_trav_starts: NaN ray, empty accel).  k_raygen runs it on the primary ray it has just generated and leaves the
 * result in the path's hit record for k_extend<true> to install (kz_trav_preset); kz_trav_seed runs it on a traversal's own ray.
 *
 * Installed as the best hit of a fresh traversal (t.best.t == tmax), a seed does not change the closest hit the traversal returns, so a
 * wrong or stale hint costs time, never correctness:
 *   - kz_trav_tri keeps the minimum of (t, geomID, primID) over the triangles it accepts, and kz_pluecker accepts t <= tfar
 *     inclusively, so the true closest triangle -- whose t is <= the seed's -- still becomes the best hit when it is tested, and a
 *     tie at equal t still goes to the smaller (geomID, primID);
 *   - the node step culls with cmax - cmin >= 0 = "may hit" on conservative boxes, so with tfar = the seed's t it still visits every
 *     node that holds a triangle hit at t <= tfar, the true closest one included;
 *   - if the seed is the closest triangle itself, its t, u, v must be the bits the traversal computes for it.  They are: the vertices
 *     are read from the shading records (KzVertex px|py|pz through the index record), which are the very floats, in the very order,
 *     that the accel's 48-byte triangle record was gathered from (k_gather_tris, KzHostScene::flatten; both builders copy them
 *     unchanged), and the test is the same kz_pluecker with the same tnear (the ray's tmin) and tfar (the ray's tmax).  k_raygen tests
 *     the very ray bits it stores, and k_extend<true> traverses the bits it loads back. */
KZ_HD bool kz_seed_hit(const KzScene &sc, float ox, float oy, float oz, float dx, float dy, float dz, float tmin, float tmax,
                       uint32_t geom, uint32_t prim, KzHit &h) {
    if (geom >= sc.n_meshes || !kz_trav_starts(sc, ox, oy, oz, dx, dy, dz, tmin, tmax)) return false;
    const KzMeshRec &m = sc.meshes[geom];
    if (prim >= m.n_triangles) return false;
    const KzU4 ix = kz_load_u4(sc.indices + (m.index_offset + prim));
    const KzVertex *vb = sc.vertices + m.vertex_offset;
    const KzU4 a = kz_load_u4(vb + ix.x), b = kz_load_u4(vb + ix.y), c = kz_load_u4(vb + ix.z);      /* px, py, pz, (u: unused) */
    if (!kz_pluecker(ox, oy, oz, dx, dy, dz, tmin, tmax, a, b, c, h.t, h.u, h.v)) return false;
    h.geom = geom; h.prim = prim;
    return true;
}
/* Presets the best hit of a freshly initialised traversal with a seed hit (kz_seed_hit on the same ray); returns true if it did.  An
 * invalid hit, or a traversal that kz_trav_init made an immediate miss, leaves the traversal as it was. */
KZ_HD bool kz_trav_preset(KzTrav &t, const KzHit &h) {
    if (h.geom == KZ_INVALID_ID || t.ng_y == 0u) return false;
    t.best = h;
    return true;
}
/* Seeds a freshly initialised traversal with a hint (kz_seed_hit on its ray, then kz_trav_preset); returns true if the ray hit it. */
KZ_HD bool kz_trav_seed(const KzScene &sc, KzTrav &t, uint32_t geom, uint32_t prim) {
    KzHit h;
    return kz_seed_hit(sc, t.ox, t.oy, t.oz, t.dx, t.dy, t.dz, t.tmin, t.best.t, geom, prim, h) && kz_trav_preset(t, h);
}

/* The plain per-ray loop.  `stk` gives the shared-memory short stack on the device; on the host
 * everything lives in the local array.  any_hit: return at the first accepted hit.  (seed_geom, seed_prim): optional hint for the
 * closest hit (kz_trav_seed). */
KZ_HD KzHit kz_trace(const KzScene &sc, const KzStackRef &stk, float ox, float oy, float oz, float dx, float dy, float dz,
                     float tmin, float tmax, bool any_hit, uint32_t seed_geom = KZ_INVALID_ID, uint32_t seed_prim = KZ_INVALID_ID) {
    KzTrav t;
    KzLocalStack ls;
    kz_trav_init(sc, t, ox, oy, oz, dx, dy, dz, tmin, tmax);
    if (sc.n_nodes == 0) return t.best;
    if (!any_hit) kz_trav_seed(sc, t, seed_geom, seed_prim);     /* an any-hit query would stop at the seed */
    for (;;) {
        if (t.ng_y > 0x00FFFFFFu) kz_trav_node(sc, t, stk, ls);
        while (t.tg_y != 0u) {
            kz_trav_tri(sc, t);
            if (any_hit && t.best.geom != KZ_INVALID_ID) return t.best;
        }
        if (t.ng_y <= 0x00FFFFFFu) {
            if (t.sp == 0) break;
            kz_trav_pop(t, stk, ls);
        }
    }
    return t.best;
}

#endif
