/* kz_common.h -- portability shims + small vector math for the sm_100a device code.
 *
 * Every per-item routine of the hot path (traversal, sampler, shading, path logic) is a
 * KZ_HD function so that tests/hostemu can compile the SAME source with g++ and check it
 * against the oracle on a box without a GPU.  The product only ever runs the __global__
 * wrappers in kz_kernels.cu; nothing here is a CPU fallback. */
#ifndef KZ_COMMON_H
#define KZ_COMMON_H
#include <stdint.h>
#include <math.h>
#include <string.h>

#if defined(__CUDACC__)
#define KZ_HD __host__ __device__ __forceinline__
#define KZ_HD_NOINLINE __host__ __device__ __noinline__
#else
#define KZ_HD inline
#define KZ_HD_NOINLINE inline
#endif

#if defined(__CUDA_ARCH__)
#define KZ_DEVICE_CODE 1
#else
#define KZ_DEVICE_CODE 0
#endif

/* ---- exactly rounded scalar ops (never contracted): used where bit parity is contracted
 *      (triangle test, hit t) ------------------------------------------------------------- */
#if KZ_DEVICE_CODE
KZ_HD float kz_fma(float a, float b, float c) { return __fmaf_rn(a, b, c); }
KZ_HD float kz_mul(float a, float b) { return __fmul_rn(a, b); }
KZ_HD float kz_add(float a, float b) { return __fadd_rn(a, b); }
KZ_HD float kz_sub(float a, float b) { return __fsub_rn(a, b); }
KZ_HD float kz_rcp(float a) { return __frcp_rn(a); }
KZ_HD float kz_div(float a, float b) { return __fdiv_rn(a, b); }
KZ_HD float kz_sqrt(float a) { return __fsqrt_rn(a); }
KZ_HD uint32_t kz_bfind(uint32_t x) { uint32_t r; asm("bfind.u32 %0, %1;" : "=r"(r) : "r"(x)); return r; }
KZ_HD uint32_t kz_popc(uint32_t x) { return (uint32_t)__popc(x); }
/* PTX prmt in its generic mode: selector nibble bit 3 replicates the sign of the selected byte
 * (the __byte_perm intrinsic only honours the low three selector bits, so it cannot be used). */
KZ_HD uint32_t kz_byte_perm(uint32_t a, uint32_t b, uint32_t s) {
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(s));
    return r;
}
KZ_HD float kz_u2f(uint32_t u) { return __uint_as_float(u); }
KZ_HD uint32_t kz_f2u(float f) { return __float_as_uint(f); }
/* prmt with an immediate selector */
#define kz_byte_perm_sel(a, b, sel) ([&] { uint32_t r_; asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r_) : "r"((uint32_t)(a)), "r"((uint32_t)(b)), "n"(sel)); return r_; }())
/* (m << 1) | sign bit of f: one funnel shift */
KZ_HD uint32_t kz_shl1_sign(uint32_t m, float f) { return __funnelshift_l(__float_as_uint(f), m, 1); }
#else
/* host emulation: volatile stops g++ from contracting a*b+c behind our back */
KZ_HD float kz_fma(float a, float b, float c) { return fmaf(a, b, c); }
KZ_HD float kz_mul(float a, float b) { volatile float r = a * b; return r; }
KZ_HD float kz_add(float a, float b) { volatile float r = a + b; return r; }
KZ_HD float kz_sub(float a, float b) { volatile float r = a - b; return r; }
KZ_HD float kz_rcp(float a) { volatile float r = 1.0f / a; return r; }
KZ_HD float kz_div(float a, float b) { volatile float r = a / b; return r; }
KZ_HD float kz_sqrt(float a) { return sqrtf(a); }
KZ_HD uint32_t kz_bfind(uint32_t x) { return 31u - (uint32_t)__builtin_clz(x); }
KZ_HD uint32_t kz_popc(uint32_t x) { return (uint32_t)__builtin_popcount(x); }
KZ_HD uint32_t kz_byte_perm(uint32_t a, uint32_t b, uint32_t s) {
    uint64_t v = ((uint64_t)b << 32) | a;
    uint32_t r = 0;
    for (int i = 0; i < 4; ++i) {
        uint32_t sel = (s >> (4 * i)) & 0xF;
        uint32_t byte = (uint32_t)((v >> (8 * (sel & 7))) & 0xFF);
        if (sel & 8) byte = (byte & 0x80) ? 0xFF : 0x00;
        r |= byte << (8 * i);
    }
    return r;
}
KZ_HD float kz_u2f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
KZ_HD uint32_t kz_f2u(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
KZ_HD uint32_t kz_shl1_sign(uint32_t m, float f) { return (m << 1) | (kz_f2u(f) >> 31); }
#define kz_byte_perm_sel(a, b, sel) kz_byte_perm((a), (b), (sel))
#endif

#define KZ_PI 3.14159265358979323846f
#define KZ_INV_PI 0.31830988618379067154f
#define KZ_EPSILON 1e-5f
#define KZ_ONE_MINUS_EPS 0x1.fffffep-1f
#define KZ_INF kz_u2f(0x7f800000u)

struct kz3 { float x, y, z; };
struct kz2 { float x, y; };

KZ_HD kz3 mk3(float x, float y, float z) { kz3 r; r.x = x; r.y = y; r.z = z; return r; }
KZ_HD kz3 mk3(float a) { return mk3(a, a, a); }
KZ_HD kz2 mk2(float x, float y) { kz2 r; r.x = x; r.y = y; return r; }
KZ_HD kz3 operator+(kz3 a, kz3 b) { return mk3(a.x + b.x, a.y + b.y, a.z + b.z); }
KZ_HD kz3 operator-(kz3 a, kz3 b) { return mk3(a.x - b.x, a.y - b.y, a.z - b.z); }
KZ_HD kz3 operator-(kz3 a) { return mk3(-a.x, -a.y, -a.z); }
KZ_HD kz3 operator*(kz3 a, kz3 b) { return mk3(a.x * b.x, a.y * b.y, a.z * b.z); }
KZ_HD kz3 operator*(kz3 a, float s) { return mk3(a.x * s, a.y * s, a.z * s); }
KZ_HD kz3 operator*(float s, kz3 a) { return mk3(s * a.x, s * a.y, s * a.z); }
#if KZ_DEVICE_CODE
/* shading vectors only (image parity is statistical): one reciprocal + three multiplies instead of three IEEE divisions */
KZ_HD kz3 operator/(kz3 a, float s) { const float r = 1.0f / s; return mk3(a.x * r, a.y * r, a.z * r); }
#else
KZ_HD kz3 operator/(kz3 a, float s) { return mk3(a.x / s, a.y / s, a.z / s); }
#endif
KZ_HD kz3 operator/(kz3 a, kz3 b) { return mk3(a.x / b.x, a.y / b.y, a.z / b.z); }
KZ_HD kz3 &operator+=(kz3 &a, kz3 b) { a = a + b; return a; }
KZ_HD kz3 &operator-=(kz3 &a, kz3 b) { a = a - b; return a; }
KZ_HD kz3 &operator*=(kz3 &a, kz3 b) { a = a * b; return a; }
KZ_HD float dot(kz3 a, kz3 b) { return a.x * b.x + (a.y * b.y + a.z * b.z); }     /* Eigen's unrolled reduction order, see oracle/kzo_math.h */
KZ_HD kz3 cross(kz3 a, kz3 b) { return mk3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
KZ_HD float sqnorm(kz3 a) { return dot(a, a); }
KZ_HD float norm(kz3 a) { return sqrtf(sqnorm(a)); }
#if KZ_DEVICE_CODE
KZ_HD kz3 normalized(kz3 a) { const float z = sqnorm(a); const float r = rsqrtf(z); return z > 0.f ? mk3(a.x * r, a.y * r, a.z * r) : a; }
#else
KZ_HD kz3 normalized(kz3 a) { float z = sqnorm(a); return z > 0.f ? a / sqrtf(z) : a; }
#endif
KZ_HD float maxcoeff(kz3 a) { return fmaxf(a.x, fmaxf(a.y, a.z)); }
KZ_HD bool iszero(kz3 a) { return a.x == 0.f && a.y == 0.f && a.z == 0.f; }
KZ_HD bool isnan3(kz3 a) { return isnan(a.x) || isnan(a.y) || isnan(a.z); }
KZ_HD float sqr(float x) { return x * x; }
KZ_HD float clampf(float v, float lo, float hi) { return v < lo ? lo : (v > hi ? hi : v); }
KZ_HD float lerpf(float t, float a, float b) { return (1.f - t) * a + t * b; }

/* common.cpp:436-445 */
KZ_HD void coordinate_system(kz3 a, kz3 &b, kz3 &c) {
    if (fabsf(a.x) > fabsf(a.y)) {
        float invLen = 1.0f / sqrtf(a.x * a.x + a.z * a.z);
        c = mk3(a.z * invLen, 0.0f, -a.x * invLen);
    } else {
        float invLen = 1.0f / sqrtf(a.y * a.y + a.z * a.z);
        c = mk3(0.0f, a.z * invLen, -a.y * invLen);
    }
    b = cross(c, a);
}
/* frame.h:13-44 */
struct KzFrame {
    kz3 s, t, n;
};
KZ_HD KzFrame frame_from_normal(kz3 n) { KzFrame f; f.n = n; coordinate_system(n, f.s, f.t); return f; }
KZ_HD kz3 to_local(const KzFrame &f, kz3 v) { return mk3(dot(v, f.s), dot(v, f.t), dot(v, f.n)); }
KZ_HD kz3 to_world(const KzFrame &f, kz3 v) { return f.s * v.x + f.t * v.y + f.n * v.z; }
KZ_HD kz3 reflect3(kz3 wi, kz3 n) { return 2 * dot(n, wi) * n - wi; }   /* common.cpp:536-538 */
KZ_HD float luminance(kz3 c) { return c.x * 0.212671f + c.y * 0.715160f + c.z * 0.072169f; }
KZ_HD float srgb_to_linear1(float v) { return v <= 0.04045f ? v * (1.0f / 12.92f) : powf((v + 0.055f) * (1.0f / 1.055f), 2.4f); }
/* toSRGB (color.h) as the reference rounds it, for the resolve's 8-bit codes: the product is rounded before the subtraction (a
 * contracted FFMA changes the code of some linear values), and the power is the double one rounded once, which gives glibc
 * powf's code on all of (0.0031308, 1].  Runs once per pixel of a resolved frame, never in a render. */
KZ_HD float linear_to_srgb1(float v) {
    return v <= 0.0031308f ? kz_mul(12.92f, v) : kz_sub(kz_mul(1.0f + 0.055f, (float)pow((double)v, (double)(1.0f / 2.4f))), 0.055f);
}
KZ_HD bool color_valid(kz3 c) {   /* common.cpp:384-391 */
    return !(c.x < 0 || !isfinite(c.x) || c.y < 0 || !isfinite(c.y) || c.z < 0 || !isfinite(c.z));
}

#endif
