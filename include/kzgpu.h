/*
 * kzgpu.h -- C ABI of the B200-native render hot path of nano-kazen.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++ types, no
 * exceptions, caller-owned host memory.  Every entry point replaces one
 * reference interface (file:line relative to the nano-kazen source tree):
 *
 *   kzgpu_scene_upload   <- Scene::addChild / Scene::activate       (src/kazen/scene.cpp:29-52,81-126)
 *                           Accel::addMesh                           (src/kazen/accel.cpp:21-23)
 *   kzgpu_accel_build    <- Accel::build (Embree BVH build)          (src/kazen/accel.cpp:25-61)
 *   kzgpu_trace[_device] <- Accel::rayIntersect core, rtcIntersect1  (src/kazen/accel.cpp:63-110)
 *                           Scene::rayIntersect / rayOccluded        (include/kazen/scene.h:79-105)
 *   kzgpu_sample_dump    <- Sampler::generateSample/next1D/next2D/nextPixel2D
 *                                                                    (src/kazen/sampler.cpp:81-390)
 *   kzgpu_render[_device]<- renderer::render -> renderBlock -> renderSample -> PathMisIntegrator::Li
 *                           -> ImageBlock::put                       (src/kazen/renderer.cpp:20-136,
 *                                                                     src/kazen/integrator.cpp:185-355,
 *                                                                     src/kazen/block.cpp:56-85)
 *   kzgpu_resolve        <- ImageBlock::toBitmap + Color3f::toSRGB   (src/kazen/block.cpp:39-45,
 *                                                                     src/kazen/common.cpp:352-366,
 *                                                                     src/kazen/bitmap.cpp:46-54)
 *
 * All functions return KZ_OK (0) or a negative error code; the message of the
 * last failure is available through kzgpu_last_error().  There is no CPU
 * fallback: kzgpu_create() fails with KZ_ERR_NO_DEVICE when no sm_100 class
 * CUDA device is usable.
 *
 * The oracle (oracle/) exposes the same functions with the prefix kzo_ over the
 * same POD tables so that tests feed byte-identical inputs to both sides.
 */
#ifndef KZGPU_H
#define KZGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ status */
#define KZ_OK                0
#define KZ_ERR_INVALID      -1   /* bad argument / malformed scene table          */
#define KZ_ERR_NO_DEVICE    -2   /* no usable CUDA device (no CPU fallback exists) */
#define KZ_ERR_CUDA         -3   /* CUDA runtime error, see kzgpu_last_error       */
#define KZ_ERR_STATE        -4   /* call order violated (e.g. trace before build)  */
#define KZ_ERR_NOMEM        -5
#define KZ_ERR_UNSUPPORTED  -6   /* plugin type outside the hot-path scope         */

#define KZ_INVALID_ID 0xFFFFFFFFu /* RTC_INVALID_GEOMETRY_ID analogue              */

/* ------------------------------------------------------------- ray batches */
/* RTCRay subset filled at accel.cpp:73-84 (mask=-1, flags=0 are implied). */
typedef struct kz_ray {
    float o[3];
    float tmin;   /* Ray3f::mint */
    float d[3];
    float tmax;   /* Ray3f::maxt */
} kz_ray;         /* 32 bytes */

/* RTCHit subset read back at accel.cpp:99-109. Miss: geom_id == KZ_INVALID_ID. */
typedef struct kz_hit {
    float    t;        /* rayhit.ray.tfar                              */
    float    u, v;     /* rayhit.hit.u / .v (P = (1-u-v) p0 + u p1 + v p2) */
    uint32_t prim_id;  /* face index inside the mesh (OBJ face order)  */
    uint32_t geom_id;  /* mesh index in scene order (accel.cpp:40-53)  */
} kz_hit;              /* 20 bytes */

/* --------------------------------------------------------------- scene POD */
/* Mesh buffers exactly as Mesh holds them (mesh.h:175-178): column-major
 * Eigen matrices == packed xyz / uv / index triples. normals/uvs may be NULL.
 * The arrays are copied to HBM as they are and turned into the renderer's records
 * there; each pointer may be a host pointer or a CUDA device pointer (arrays that
 * were produced on a GPU are read in place). */
typedef struct kz_mesh_desc {
    const float    *positions;   /* 3 * n_vertices  */
    const float    *normals;     /* 3 * n_vertices or NULL */
    const float    *uvs;         /* 2 * n_vertices or NULL */
    const uint32_t *indices;     /* 3 * n_triangles */
    uint32_t        n_vertices;
    uint32_t        n_triangles;
    int32_t         bsdf;        /* index into kz_scene_desc.bsdfs              */
    int32_t         light;       /* index into kz_scene_desc.lights, -1 = none  */
} kz_mesh_desc;

/* Texture expression nodes (texture.cpp:10-270). */
enum kz_texture_type {
    KZ_TEX_CONSTANT   = 0,  /* "constanttexture": color                         */
    KZ_TEX_IMAGE      = 1,  /* "imagetexture": image, scale, srgb               */
    KZ_TEX_BACKGROUND = 2,  /* "background": a * child[0] (a = intensity)       */
    KZ_TEX_COLORRAMP  = 3,  /* "colorramp": a + (b-a)*clamp01(child[0])         */
    KZ_TEX_BLEND      = 4   /* "blend": child = {mask,input1,input2}; mode      */
};
#define KZ_BLEND_MIX      0
#define KZ_BLEND_MULTIPLY 1
#define KZ_BLEND_OTHER    2  /* unknown blendmode string -> 0 (texture.cpp:229) */

typedef struct kz_texture_desc {
    int32_t type;
    float   color[3];     /* CONSTANT                                           */
    int32_t image;        /* IMAGE: index into images                           */
    float   scale;        /* IMAGE                                              */
    int32_t srgb;         /* IMAGE: colorspace == "srgb" -> toLinearRGB         */
    float   a, b;         /* BACKGROUND: a=intensity; COLORRAMP: a=min,b=max    */
    int32_t mode;         /* BLEND                                              */
    int32_t child[3];     /* node indices, -1 = absent (defaults texture.cpp:215-217) */
} kz_texture_desc;

/* Decoded image, row 0 = first scanline of the file, linear float, 3 channels. */
typedef struct kz_image_desc {
    int32_t      width, height;
    const float *rgb;     /* 3 * width * height */
} kz_image_desc;

enum kz_bsdf_type {
    KZ_BSDF_DIFFUSE         = 0,  /* "diffuse"          bsdf.cpp:20-92     */
    KZ_BSDF_KISS            = 1,  /* "kazenstandard"    bsdf.cpp:1157-1418 */
    KZ_BSDF_NORMALMAP       = 2,  /* "normalmap"        bsdf.cpp:281-417   */
    /* SURVEY 8(f)-1: the remaining BSDF plugins */
    KZ_BSDF_DIELECTRIC      = 3,  /* "dielectric"       bsdf.cpp:98-156    */
    KZ_BSDF_MIRROR          = 4,  /* "mirror"           bsdf.cpp:162-196   */
    KZ_BSDF_LAMBERTIAN      = 5,  /* "lambertian"       bsdf.cpp:202-276   */
    KZ_BSDF_GGX             = 6,  /* "ggx"              bsdf.cpp:629-690   */
    KZ_BSDF_ROUGHCONDUCTOR  = 7,  /* "roughconductor"   bsdf.cpp:693-812   */
    KZ_BSDF_ROUGHPLASTIC    = 8,  /* "roughplastic"     bsdf.cpp:815-944   */
    KZ_BSDF_ROUGHDIELECTRIC = 9   /* "roughdielectric"  bsdf.cpp:947-1145  */
};

typedef struct kz_bsdf_desc {
    int32_t type;
    float   albedo[3];                           /* DIFFUSE albedo; ROUGHPLASTIC kd */
    int32_t base_color, roughness, metallic;     /* KISS: texture node indices; LAMBERTIAN/GGX: base_color = albedo texture */
    float   anisotropy, specular, specular_tint; /* KISS scalars bsdf.cpp:1159-1167; GGX: anisotropy */
    float   clearcoat, clearcoat_roughness;
    float   sheen, sheen_tint;
    int32_t normal_map;                          /* NORMALMAP: texture node       */
    int32_t nested;                              /* NORMALMAP: bsdf index         */
    float   int_ior, ext_ior;                    /* DIELECTRIC, ROUGHPLASTIC, ROUGHDIELECTRIC */
    float   alpha;                               /* ROUGHCONDUCTOR/ROUGHPLASTIC/ROUGHDIELECTRIC: max(1e-3, roughness^2); GGX: roughness as given */
    float   eta[3], k[3];                        /* ROUGHCONDUCTOR complex IOR (bsdf.cpp:703-714) */
} kz_bsdf_desc;

/* AreaLight (light.cpp:7-66); radiance = intensity * color. */
typedef struct kz_light_desc {
    float   radiance[3];
    int32_t primary_visibility;   /* lightPrimaryVisibility, default 0 */
} kz_light_desc;

enum kz_camera_type { KZ_CAM_PERSPECTIVE = 0, KZ_CAM_THINLENS = 1 };

/* Camera after activate() (camera.cpp:35-68,156-189). Matrices are row-major. */
typedef struct kz_camera_desc {
    int32_t type;
    int32_t width, height;
    float   sample_to_camera[16];
    float   camera_to_world[16];
    float   near_clip, far_clip;
    float   aperture_radius, focus_distance;   /* thinlens only */
} kz_camera_desc;

enum kz_sampler_type {
    KZ_SAMPLER_INDEPENDENT = 0,
    KZ_SAMPLER_STRATIFIED  = 1,
    KZ_SAMPLER_CORRELATED  = 2,
    KZ_SAMPLER_PMJ02BN     = 3
};

/* Sampler after construction (sampler.cpp:20-22,83-93,178-189,275-315):
 * sample_count is already rounded the way the constructor rounds it. */
typedef struct kz_sampler_desc {
    int32_t  type;
    uint32_t sample_count;
    uint64_t seed;
    int32_t  res_x, res_y;          /* stratified: res_x=res_y=resolution; correlated: m_resolution */
    /* pmj02bn tables (missing from the reference mount). NULL -> kzgpu uses the
     * documented fallback generator (NOT pbrt's table; parity unpinned).        */
    const uint16_t *blue_noise;     /* [48][128][128]           */
    const uint32_t *pmj02bn;        /* [5][65536][2]            */
} kz_sampler_desc;

enum kz_integrator_type {
    KZ_INTEGRATOR_PATH_MIS  = 0,   /* "path_mis"   integrator.cpp:185-355 (the hot path)         */
    KZ_INTEGRATOR_NORMALS   = 1,   /* "normals"    integrator.cpp:11-34   (SURVEY 8f-3)          */
    KZ_INTEGRATOR_AO        = 2,   /* "ao"         integrator.cpp:37-70                          */
    KZ_INTEGRATOR_WHITTED   = 3,   /* "whitted"    integrator.cpp:74-134                         */
    KZ_INTEGRATOR_PATH_MATS = 4    /* "path_mats"  integrator.cpp:137-181                        */
};

/* PathMisIntegrator properties (integrator.cpp:187-193); the other integrators have none. */
typedef struct kz_integrator_desc {
    int32_t max_depth;
    float   trace_bias;
    int32_t regularization;
    float   accumulated_roughness;
    int32_t type;                  /* kz_integrator_type */
    /* path_mis only ("envSampling", default 0 = the reference estimator): 1 also samples the background as a light.  Next-event
     * estimation then picks the environment with probability 1 / (emitters + 1) and draws a direction from a luminance table of the
     * background (built on the GPU at kzgpu_scene_upload), and a BSDF-sampled ray that escapes is weighted by the power heuristic
     * against that density.  The estimate is unbiased either way; with an HDR sky whose light comes from a small bright region (a sun,
     * a window) it converges much faster.  Nothing changes when the background is absent or black in every direction (no
     * background, zero intensity, colorramp / blend chains, an all-black image), nor for the other integrators. */
    int32_t env_sampling;
    /* path_mis only ("textureFiltering", default 0 = every texture lookup reads mip level 0, as the reference does): 1 filters image
     * textures by their screen footprint.  Every image then gets its full mip pyramid resident in HBM (built on the GPU at
     * kzgpu_scene_upload; about a third more texels), and a uv-mode lookup of a texture a BSDF reads (kazenstandard baseColor /
     * roughness / metallic, a normal map, the lambertian / ggx albedo) is a trilinear lookup at the level of the footprint: bicubic at
     * the two levels around it, lerped; level 0 exactly when the texture is magnified.  The footprint is pbrt-v4's camera estimate
     * (uv derivatives at the hit from the camera alone, scaled by max(1/8, 1/sqrt(sample_count))), so far-away and grazing textures
     * stop aliasing and converge at low sample counts.  It does not follow the path: after a bounce the lookup is as sharp as the
     * camera would see that point.  Background lookups always read level 0.  Nothing changes when no such texture reads an image,
     * nor for the other integrators. */
    int32_t texture_filtering;
} kz_integrator_desc;

/* Reconstruction filter tabulated as ImageBlock does (block.cpp:13-21). */
typedef struct kz_filter_desc {
    float radius;
    float table[33];   /* KAZEN_FILTER_RESOLUTION + 1, table[32] = 0 */
} kz_filter_desc;

typedef struct kz_scene_desc {
    const kz_mesh_desc    *meshes;    uint32_t n_meshes;
    const kz_bsdf_desc    *bsdfs;     uint32_t n_bsdfs;
    const kz_texture_desc *textures;  uint32_t n_textures;
    const kz_image_desc   *images;    uint32_t n_images;
    const kz_light_desc   *lights;    uint32_t n_lights;
    int32_t                background;  /* texture node with id="background", -1 = none */
    kz_camera_desc         camera;
    kz_sampler_desc        sampler;
    kz_integrator_desc     integrator;
    kz_filter_desc         filter;
} kz_scene_desc;

/* --------------------------------------------------------------- rendering */
/* One call renders sample indices [spp_begin, spp_end) of every pixel of the
 * rectangle [x0,x1) x [y0,y1) and ADDS the filtered splats into the bordered
 * frame (block.cpp:56-85).  With the pmj02bn sampler spp_end must not exceed the
 * sampler's sample_count (its per-pixel tables hold sample_count entries).  Frame layout: (H+2b) rows of (W+2b) float4
 * (r*w, g*w, b*w, w), b = ceil(radius - 0.5).  Sharding across GPUs = disjoint
 * spp ranges / rectangles followed by a sum of the frames. */
typedef struct kz_render_req {
    int32_t x0, y0, x1, y1;
    int32_t spp_begin, spp_end;
    int32_t clear_frame;      /* 1: zero the frame first */
} kz_render_req;

typedef struct kz_stats {
    uint64_t paths;            /* renderSample invocations                          */
    uint64_t rays_extension;   /* primary + re-trace + extension closest-hit queries */
    uint64_t rays_shadow;      /* shadow segments (incl. light-stepping re-traces)   */
    uint64_t vertices;         /* shaded path vertices                               */
    uint64_t kernel_launches;  /* CUDA kernels launched by this context since reset  */
    double   ms_trace;         /* device time in traversal kernels                   */
    double   ms_shade;         /* device time in raygen/shade/accumulate kernels     */
    double   ms_total;         /* device time of the render calls since reset (accumulates) */
    uint64_t bvh_nodes;        /* wide nodes                                         */
    uint64_t bvh_bytes;        /* nodes + leaf triangles                             */
    double   ms_build;         /* wall time of the last kzgpu_accel_build (host + device) */
    double   ms_upload;        /* wall time of the last kzgpu_scene_upload           */
    double   ms_merge;         /* device time in the multi-device frame merge since reset */
    uint64_t rays_seeded;      /* primary rays whose traversal started from their pixel's previous hit (the "primary_hint" option) */
} kz_stats;

#define KZ_BUILD_HOST_SAH 0    /* binned SAH on the host, collapsed to 8-wide, uploaded */
#define KZ_BUILD_LBVH     1    /* on-GPU Morton LBVH, collapsed to 8-wide               */
/* On-GPU LBVH whose subtrees never mix meshes: every slot of every node holds triangles of exactly one mesh, or whole meshes only (so no
 * leaf slot holds two meshes).  The references are sorted by mesh first (meshes ranked by the Morton code of their box centres), then by
 * Morton code, and not pre-split.  A fresh build traces as fast as KZ_BUILD_LBVH or up to ~10 % slower where meshes overlap, but when meshes move rigidly
 * (kzgpu_mesh_transform) each mesh's subtrees move with it, so kzgpu_accel_refit keeps their boxes tight and only the few nodes above the
 * meshes grow.  Build with it when whole meshes move from frame to frame and refit; DESIGN.md section 7 has measurements. */
#define KZ_BUILD_LBVH_MESHES 2

typedef struct kzgpu_ctx kzgpu_ctx;

int  kzgpu_create(const int *device_ids, int n_devices, kzgpu_ctx **out);
void kzgpu_destroy(kzgpu_ctx *ctx);
const char *kzgpu_last_error(const kzgpu_ctx *ctx);   /* ctx may be NULL: global message */

int  kzgpu_scene_upload(kzgpu_ctx *ctx, const kz_scene_desc *scene);
int  kzgpu_accel_build(kzgpu_ctx *ctx, int builder);

/* Animation: change an uploaded scene in place, then refit its accel instead of uploading and building again.
 * Like kzgpu_scene_upload and kzgpu_accel_build, these calls require that everything enqueued with kzgpu_render_device
 * or kzgpu_trace_device has finished (synchronise the stream first); they do not wait for it themselves. */

/* Replaces the vertex positions of mesh `mesh` of the uploaded scene, and its normals if `normals` != NULL.
 * Each array holds 3 * n_vertices floats, laid out as in kz_mesh_desc, and may be a host or a device pointer.
 * Topology, uvs, materials and lights are unchanged; an emitter's area CDF and the bounds of the invisible emitters
 * are recomputed.  Passing normals for a mesh uploaded without normals is KZ_ERR_INVALID; an invalid call changes nothing.
 * Entry points that need the accel return KZ_ERR_STATE until kzgpu_accel_refit or kzgpu_accel_build has run.
 * The primary-hit hints are kept: any hint yields the same hits, and those of the last frame are the best guess. */
int  kzgpu_mesh_update(kzgpu_ctx *ctx, int mesh, const float *positions, const float *normals);

/* Sets mesh `mesh`'s positions to matrix * p and, if it has normals, its normals to normalize(inverse^T * n), where p and n are the
 * mesh's rest pose: the arrays of the upload or of the last kzgpu_mesh_update of this mesh (so transforming twice does not compose).
 * matrix and inverse are row-major 4x4, as kz_camera_desc's; inverse may be NULL for a mesh without normals.  The arithmetic is the
 * C++ host's `toWorld` (Transform::point divides by w; normals are normalised as the OBJ loader does), rounded the same way, so a mesh
 * placed here equals the same OBJ loaded with that transform, bit for bit.  It runs on every device; the rest pose is kept in HBM for
 * meshes that have been transformed (12 bytes per vertex, 24 with normals) until the next kzgpu_scene_upload.  An emitter's area CDF and
 * the bounds of the invisible emitters are recomputed.  A NULL matrix, a NULL inverse for a mesh with normals, a non-finite entry or a
 * mesh index out of range is KZ_ERR_INVALID; an invalid call changes nothing.  As after kzgpu_mesh_update, entry points that need the
 * accel return KZ_ERR_STATE until kzgpu_accel_refit or kzgpu_accel_build has run. */
int  kzgpu_mesh_transform(kzgpu_ctx *ctx, int mesh, const float matrix[16], const float inverse[16]);

/* Refits the built accel to the current vertex positions on every device of the context.
 * The tree is the same; the boxes, triangle records and traversal slack are recomputed, so trace and render return
 * exactly what a fresh build over the new positions returns (the tree only decides how fast).  A tree built for very
 * different positions traces slower: rebuild when the motion is large (DESIGN.md section 7 has measurements).
 * Returns when done, like kzgpu_accel_build.  KZ_ERR_STATE if no accel was built since the last upload. */
int  kzgpu_accel_refit(kzgpu_ctx *ctx);

/* Replaces the camera.  width/height must equal the uploaded ones (the frame and the hints are sized by them). */
int  kzgpu_camera_update(kzgpu_ctx *ctx, const kz_camera_desc *camera);

/* Parity probe: copies device `device`'s accel (n_nodes 80-byte nodes, 3 * n_tris float4) to host buffers sized from
 * kz_stats: n_nodes = bvh_nodes, n_tris = (bvh_bytes - 80 * bvh_nodes) / 48. */
int  kzgpu_accel_dump(kzgpu_ctx *ctx, int device, void *nodes, void *tris);

/* Closest-hit queries on host buffers (H2D + trace + D2H), shadow=1 uses the
 * shadow-ray variant of accel.cpp:100-104 (same closest-hit, u/v/prim still filled). */
int  kzgpu_trace(kzgpu_ctx *ctx, int device, const kz_ray *rays, size_t n, int shadow, kz_hit *hits);
/* Same on device-resident buffers of `device`; runs on `stream` (cudaStream_t as void*, NULL = default).
 * d_rays must be 16-byte aligned (rays are read as two 128-bit loads), d_hits 4-byte aligned. */
int  kzgpu_trace_device(kzgpu_ctx *ctx, int device, const void *d_rays, size_t n, int shadow,
                        void *d_hits, void *stream);
/* Shadow-ray visibility with kazen's invisible-light stepping (integrator.cpp:259-278):
 * out[i] = 1 if occluded, 0 otherwise; segments[i] = closest-hit queries issued. */
int  kzgpu_occluded(kzgpu_ctx *ctx, int device, const kz_ray *rays, size_t n, float trace_bias,
                    uint8_t *occluded, uint8_t *segments);

/* Sampler parity: for each (px,py,sampleIndex) triple run generateSample() and then
 * the draw pattern, a string over {'P' = nextPixel2D, '2' = next2D, '1' = next1D};
 * out receives the floats in draw order (2 per 'P'/'2', 1 per '1'), n_floats each. */
int  kzgpu_sample_dump(kzgpu_ctx *ctx, const int32_t *pixel_sample_triples, size_t n,
                       const char *pattern, float *out);

/* Camera parity: rays for explicit (pixelSample, apertureSample) pairs, 4 floats each. */
int  kzgpu_camera_rays(kzgpu_ctx *ctx, const float *samples4, size_t n, kz_ray *out);

/* Shading parity probe: one BSDF query in the local shading frame on the device.
 * mode 0 = BSDF::eval (out[0..2]), 1 = BSDF::pdf (out[0]), 2 = BSDF::sample (out[0..2] weight,
 * out[3..5] wo, out[6] measure, out[7] pdf).  bsdf.cpp:20-92,281-417,1215-1371. */
int  kzgpu_bsdf_query(kzgpu_ctx *ctx, int bsdf, int mode, const float wi[3], const float wo[3], const float uv[2],
                      float accumulated_roughness, float sample1, const float sample2[2], float out[8]);

/* Texture probe: periodic bicubic lookup of image `image` at mip `level` (0 = finest; the pyramid is built on the GPU by 2x2 box
 * filtering: the resident one when the scene filters its textures, otherwise a temporary one for this call) for n (s,t) pairs -> n rgb triples.  ImageTexture::eval's texture() call with zero
 * derivatives (texture.cpp:46-64) is level 0 with s = u*scale, t = (1-v)*scale. */
int  kzgpu_image_lookup(kzgpu_ctx *ctx, int image, int level, const float *st, size_t n, float *rgb);

/* Whole-frame render into a host frame ((H+2b)*(W+2b)*4 floats). Multi-device contexts
 * shard [spp_begin,spp_end) by sample index across their devices and merge the frames on
 * the devices (ImageBlock::put(ImageBlock&), block.cpp:87-96): every device sums its slice
 * of all frames through NVLink peer loads into the first device's frame, which is then
 * copied out once.  clear_frame = 0 adds to the frame passed in. */
int  kzgpu_render(kzgpu_ctx *ctx, const kz_render_req *req, float *frame_rgbw);
/* Single-device variant leaving the frame in HBM (for an NCCL reduce by the caller), enqueued on
 * `stream` without synchronising.  *d_frame_inout != NULL on entry: splat into that caller-owned
 * device buffer of (H+2b)*(W+2b) float4; NULL on entry: use the context's frame and return it. */
int  kzgpu_render_device(kzgpu_ctx *ctx, int device, const kz_render_req *req, void **d_frame_inout,
                         void *stream);
int  kzgpu_frame_dims(const kzgpu_ctx *ctx, int32_t *width, int32_t *height, int32_t *border);

/* frame -> rgb/w -> sRGB 8-bit (truncating, bitmap.cpp:49-51). Host in, host out. */
int  kzgpu_resolve(kzgpu_ctx *ctx, const float *frame_rgbw, float *rgb_linear /* W*H*3 or NULL */,
                   uint8_t *srgb8 /* W*H*3 or NULL */);

/* Post-intersection parity probe (Accel::rayIntersect's second half, accel.cpp:113-236): for each ray, trace it and fill the
 * Intersection of the closest hit.  24 floats per ray: t, mesh (as float, -1 = miss), p[3], uv[2], geoFrame.n[3],
 * shFrame.s[3], shFrame.t[3], shFrame.n[3], dpdu[3], 2 x 0. */
int  kzgpu_intersection_dump(kzgpu_ctx *ctx, const kz_ray *rays, size_t n, float *out24);

/* Emitter sampling parity probe (Scene::getRandomLight scene.h:45-56, Mesh::sample mesh.cpp:108-133, AreaLight::sample /
 * pdf / eval light.cpp:16-51): for reference point ref[i] and the five random numbers u5[i] = (light pick, triangle pick,
 * barycentric 1, barycentric 2, unused) in the order Li draws them.  16 floats per query: mesh, p[3], n[3], wi[3], dist, pdf (solid
 * angle, without the light-pick probability), Le/pdf [3], 0. */
int  kzgpu_light_sample_dump(kzgpu_ctx *ctx, const float *ref3, const float *u5, size_t n, float *out16);

/* Environment sampling probe (path_mis with env_sampling): for each pair u2[i] = (row draw, column draw) of device `device`'s
 * environment table, 8 floats: the sampled direction [3], its solid-angle density (the one the miss branch uses), the background's
 * radiance in that direction [3], 0.  KZ_ERR_STATE when the uploaded scene does not count the environment as a light. */
int  kzgpu_env_sample_dump(kzgpu_ctx *ctx, int device, const float *u2, size_t n, float *out8);

/* Texture footprint probe (texture_filtering): traces each ray on device `device` and writes 8 floats at its closest hit: mesh (as
 * float, -1 = miss), uv[2] (as the shader sees it), du/dx, dv/dx, du/dy, dv/dy (the footprint the filtered shade kernels compute
 * there, for the current camera and vertices), 0.  Runs whether or not the scene filters its textures. */
int  kzgpu_texture_footprint_dump(kzgpu_ctx *ctx, int device, const kz_ray *rays, size_t n, float *out8);

/* Filtered texture probe: the shade kernels' lookup of image `image` for n (s, t) pairs with st derivatives dst4[i] = (ds/dx, dt/dx,
 * ds/dy, dt/dy) -> n rgb triples (before sRGB linearisation), on the first device.  KZ_ERR_STATE unless the uploaded scene filters
 * its textures (the pyramids are resident only then). */
int  kzgpu_image_lookup_filtered(kzgpu_ctx *ctx, int image, const float *st, const float *dst4, size_t n, float *rgb);

/* Tuning knobs of the wavefront (defaults: up to 3 lanes -- frames below 2^25 paths use 2 --, 2^24 path slots per lane, runs of 64 sample
 * indices per pixel tile in path order; also read from KZGPU_LANES / KZGPU_POOL_LOG2 / KZGPU_SPP_GROUP at
 * kzgpu_create).  "lanes" = concurrent chunks per device (1 = strictly serial kernels, which is what per-kernel timings in
 * kz_stats need to be meaningful), "pool_log2" = log2 of the path slots per chunk, "spp_group" = consecutive sample indices of a pixel
 * tile that are neighbours in path order (1 = sample-major), "primary_hint" (KZGPU_PRIMARY_HINT) = whether a primary ray's traversal
 * starts from the triangle its pixel's previous primary ray hit: 0 = never, 1 (default) = in scenes of at least 2^20 triangles (where
 * it pays), 2 = always.  None of them changes which paths are traced or what they hit. */
int  kzgpu_configure(kzgpu_ctx *ctx, const char *key, int value);

int  kzgpu_stats(kzgpu_ctx *ctx, kz_stats *out);
int  kzgpu_stats_reset(kzgpu_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* KZGPU_H */
