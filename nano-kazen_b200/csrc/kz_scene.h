/* kz_scene.h -- HBM-resident scene layout shared by the kernels (and by tests/hostemu).
 *
 * Accel:
 *   nodes : 80-byte 8-wide compressed nodes (quantised child boxes after Ylitie/Karras/Laine 2017; the per-slot meta
 *           bytes of that layout are replaced by two masks in slot order -- imask and trimask -- so that the traversal
 *           builds its hit masks with word-parallel bit operations instead of per-child shifts), read as 5 x 16-byte loads.
 *   tris  : 48 bytes per triangle in leaf order = 3 x float4
 *           (p0.xyz | geomID), (p1.xyz | primID), (p2.xyz | 0): raw vertices because the
 *           parity-contracted Pluecker test works on origin-relative vertices.
 * Shading: per-mesh interleaved vertex records (KzVertex) and 16-byte index records concatenated, addressed through KzMeshRec.
 */
#ifndef KZ_SCENE_H
#define KZ_SCENE_H
#include "kz_common.h"
#include "../../include/kzgpu.h"

struct alignas(16) KzU4 { uint32_t x, y, z, w; };     /* 16-byte aligned: moves as one 128-bit load / store */
struct alignas(16) KzF4 { float x, y, z, w; };

struct alignas(16) KzNode8 {
    float    px, py, pz;          /* quantisation origin                                   */
    uint8_t  ex, ey, ez, imask;   /* per-axis exponent (IEEE biased), internal-child mask  */
    uint32_t child_base;          /* index of first internal child                         */
    uint32_t tri_base;            /* index of first triangle referenced by this node       */
    uint32_t trimask;             /* leaf slot s owns bits [3s, 3s+3): its n <= 3 triangles set the low n of them; the triangle of set bit k
                                     is tri_base + popc(trimask below k) (triangles are stored in slot order)                       */
    uint32_t magic;               /* KZ_NODE_MAGIC: operand of the byte->float permutes of the node step (kz_traverse.h)             */
    uint8_t  qlox[8], qloy[8], qloz[8];
    uint8_t  qhix[8], qhiy[8], qhiz[8];
};
#define KZ_NODE_MAGIC 0x47000000u
static_assert(sizeof(KzNode8) == 80, "node must be 80 bytes");

struct KzMeshRec {
    uint32_t vertex_offset;   /* into vertices */
    uint32_t index_offset;    /* into indices (in triangles)               */
    uint32_t n_triangles;
    uint32_t flags;           /* KZ_MESH_* */
    int32_t  bsdf;
    int32_t  light;
    uint32_t cdf_offset;      /* into light_cdf (n_triangles+1 floats) */
    float    inv_area;        /* DiscretePDF normalization = 1/sum(area), mesh.h pdf() */
};
#define KZ_MESH_HAS_NORMALS 1u
#define KZ_MESH_HAS_UVS 2u
#define KZ_MESH_IS_LIGHT 4u
#define KZ_MESH_LIGHT_VISIBLE 8u

/* material classes used to sort the shade queues */
#define KZ_CLASS_TERMINAL 0   /* miss or light hit */
#define KZ_CLASS_DIFFUSE 1
#define KZ_CLASS_KISS 2
#define KZ_CLASS_NORMALMAP 3
#define KZ_CLASS_GENERIC 4    /* the other BSDF plugins (SURVEY 8f-1), dispatched at run time */
#define KZ_NUM_CLASSES 5

/* All attributes of a vertex in one 32-byte record (a whole DRAM sector, two 128-bit or one 256-bit load) instead of three
 * arrays: a shaded vertex touches 3 sectors of vertex data + 1 of indices instead of up to 12. */
struct alignas(16) KzVertex { float px, py, pz, u, nx, ny, nz, v; };

struct KzImageRec {
    int32_t  width, height;
    uint32_t texel_offset;    /* float4 index of mip level 0 */
    int32_t  n_levels;        /* mip pyramid levels resident after level 0 (level l follows l-1) */
};

/* kz_integrator_desc as the kernels read it (the same layout as before env_sampling): kzgpu_scene_upload resolves env_sampling into which k_shade instantiations run */
struct KzIntegrator {
    int32_t max_depth;
    float   trace_bias;
    int32_t regularization;
    float   accumulated_roughness;
    int32_t type;
};

struct KzScene {
    /* accel */
    const KzNode8 *nodes;
    const KzF4    *tris;
    uint32_t       n_nodes, n_tris;
    float          scene_max_abs;     /* max |coordinate| of any vertex: scales the traversal slack */
    /* shading geometry */
    const KzMeshRec *meshes;
    uint32_t         n_meshes;
    const KzVertex *vertices;         /* position|u, normal|v: one 32-byte sector per vertex              */
    const KzU4     *indices;          /* i0, i1, i2, 0 per triangle: one 128-bit load                      */
    const float    *light_cdf;
    const int32_t  *light_meshes;     /* scene.cpp:42-46 order */
    int32_t         n_light_meshes;
    int32_t         n_invisible_lights;                  /* emitters a shadow ray passes through (integrator.cpp:259-294) ...  */
    float           inv_light_lo[3], inv_light_hi[3];    /* ... and the bounds of their vertices                               */
    /* materials */
    const kz_bsdf_desc    *bsdfs;
    const kz_texture_desc *textures;
    const KzImageRec      *images;
    const KzF4            *texels;
    const kz_light_desc   *lights;
    int32_t                background;
    /* render setup */
    kz_camera_desc     camera;
    KzIntegrator       integrator;
    kz_filter_desc     filter;
    int32_t            border;
    /* sampler */
    int32_t  sampler_type;
    uint32_t sample_count;
    uint64_t seed;
    int32_t  res_x, res_y;
    const uint16_t *blue_noise;
    const uint32_t *pmj02bn;
    const kz2      *pmj_pixel_samples;
    int32_t         pmj_tile_size;
};

#endif
