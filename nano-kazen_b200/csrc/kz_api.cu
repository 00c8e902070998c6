/* kz_api.cu -- the C ABI of include/kzgpu.h over the sm_100a kernels (kz_kernels.cuh).
 *
 * One kzgpu_ctx owns 1..N CUDA devices with the scene replicated on each (SURVEY 8e).  All work of
 * a call is enqueued on a stream without any host round trip (queue counts live in HBM, grids are
 * persistent), so a single host thread drives all devices of a context concurrently.
 * There is no CPU path in this file: without a usable sm_100-class device kzgpu_create fails.
 */
#include "kz_kernels.cuh"
#include "kz_host_scene.h"
#include "kz_lbvh.cuh"
#include "kz_ingest.cuh"
#include "kz_refit.cuh"
#include "kz_owner.h"
#include <cuda_runtime.h>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <memory>
#include <string>
#include <thread>
#include <vector>

namespace {

thread_local std::string g_error;

enum { CAT_TRACE = 0, CAT_SHADE = 1, CAT_TOTAL = 2, CAT_MERGE = 3, CAT_COUNT = 4 };

struct EvPair { cudaEvent_t a, b; int cat; };

#define KZ_MAX_LANES 4
struct Lane {
    Stream stream;                   /* lane 1.. only; lane 0 runs on the caller's stream */
    Event done;
    DevMem ctl_mem;
    KzControl *ctl = nullptr;
    uint32_t pool_cap = 0;
    DevMem pool[6 + KZ_NUM_CLASSES]; /* pool_cap slots each: the path state and the queues below */
    KzPathState st{};
    KzQueues q{};
};

/* A device's accel: the node and triangle arrays (KzNode8[n_nodes], KzF4[3 * n_tris]) and the max |coordinate| they were built for */
struct Accel {
    DevMem nodes, tris;
    uint32_t n_nodes = 0, n_tris = 0;
    float max_abs = 0.f;
};

struct Device {
    int id = -1;
    int sm_count = 0;
    Stream stream, copy_in, copy_out;
    std::vector<DevMem> tables;      /* scene tables and the vertex / index / texel records that sc points into */
    Accel accel;
    KzScene sc{};                    /* device pointers */
    bool has_accel = false;
    /* wavefront pools: the chunks of a render alternate between two lanes (own stream, path state, queues and control block), so
     * the ramp-up and the tail of one chunk's persistent kernels are filled by the other chunk's work */
    Lane lane[KZ_MAX_LANES];
    KzControl *ctl = nullptr;        /* = lane[0].ctl: counters of the batch entry points */
    DevMem cursor;                   /* batch-trace fetch cursor */
    DevMem frame_mem;                /* the context's own frame; frame may point at a caller's instead (kzgpu_render_device) */
    KzF4 *frame = nullptr;
    size_t frame_texels = 0;
    /* primary-hit hints (k_raygen runs the seed test, KzExtendJob<true>::seed installs it): (geomID, primID) per film pixel, allocated by the first render that uses them and
     * invalidated (all 0xFF) whenever the accel or the film may have changed -- a hint is only worth something for the same triangles */
    DevMem hint;
    bool hint_stale = true;
    Event splat_done, merge_done;    /* multi-device frame merge (k_frame_reduce) */
    /* kzgpu_accel_refit: node boxes of the level below (kept between refits), its two result words (max |coordinate| as an ordered
     * uint, a failed level check) and whether this accel's level layout was checked on this device */
    DevMem refit_boxes, refit_flags;
    bool levels_checked = false;
    /* scratch for host-pointer entry points */
    DevMem scratch[3];
    /* launch geometry */
    int grid_extend0 = 0, grid_extend = 0, grid_shadow = 0, grid_trace = 0, grid_occ = 0, grid_shade[KZ_NUM_CLASSES] = {0, 0, 0, 0, 0};
    /* timing */
    std::vector<EvPair> pending;
    std::vector<cudaEvent_t> free_events;
    double ms[CAT_COUNT] = {0, 0, 0, 0};
    uint64_t launches = 0;

    /* releases everything with this device current, after its work finished (the members go after this body) */
    ~Device() {
        if (id < 0) return;
        cudaSetDevice(id);
        cudaDeviceSynchronize();
        for (cudaEvent_t e : free_events) cudaEventDestroy(e);
    }
};

}  // namespace

struct kzgpu_ctx {
    std::vector<Device> devs;
    std::unique_ptr<KzHostScene> hs;
    bool class_present[KZ_NUM_CLASSES] = {true, false, false, false, false};
    bool uploaded = false, built = false;
    uint32_t pool_cap = 1u << 24;     /* path slots per chunk and lane (160 B each = 2.5 GiB): every launch costs ~18 us of ramp + tail, so few big chunks win */
    int lanes = 3;                    /* concurrent chunks per device at most, 1..4 (KZGPU_LANES=1: strictly serial chunks); frames below 2^25 paths use two */
    int primary_hint = 1;             /* seed primary rays with the triangle their pixel hit last (k_raygen, KzExtendJob<true>::seed; KZGPU_PRIMARY_HINT / "primary_hint"):
                                       * 0 = never, 1 = for scenes of at least KZ_HINT_MIN_TRIS triangles, 2 = always.  Measured on B200, Mpaths/s off -> on:
                                       * 10^8-triangle 4K headline 909 -> 975 (primary pass ~25 % shorter); WarmStudio.xml 1292 -> 1269, configs[2] 873 -> 866,
                                       * configs[3] 849 -> 838 (few triangles: the primaries are cheap, the extra loads and spills of the seed are not) */
    int spp_group = 64;               /* sample indices of one tile that are neighbours in path order (KZGPU_SPP_GROUP, 1 = sample-major).  Measured on the
                                       * 10^8-triangle 4K headline / WarmStudio.xml / configs[2], Mpaths/s, with k_accumulate splatting one 32-path unit per warp at a time
                                       * (the splats of neighbouring warps then pile onto the same texels): 1 -> 827 / 1213 / 821, 8 -> 842 / 1213 / 823, 64 -> 807 / 1110 / 780;
                                       * with every warp of k_accumulate walking its own run of units: 8 -> 892 / 1261 / 860, 16 -> 904 / 1262 / 861,
                                       * 32 -> 909 / 1264 / 862, 64 -> 918 / 1263 / 866 */
    kz_stats totals{};
    double ms_build = 0;
    uint64_t bvh_nodes = 0, bvh_bytes = 0;
    double last_total_ms = 0;
    double ms_upload = 0;             /* wall time of the last kzgpu_scene_upload */
    std::vector<uint32_t> levels;     /* wide-tree level l of the built accel = nodes [levels[l], levels[l + 1]); empty: not laid out by level */
    std::string error;
};

namespace {

int fail(kzgpu_ctx *ctx, int code, const std::string &msg) {
    g_error = msg;
    if (ctx) ctx->error = msg;
    return code;
}

#define KZ_CUDA(ctx, call)                                                                                   \
    do {                                                                                                     \
        cudaError_t e__ = (call);                                                                            \
        if (e__ != cudaSuccess)                                                                              \
            return fail(ctx, e__ == cudaErrorMemoryAllocation ? KZ_ERR_NOMEM : KZ_ERR_CUDA,                  \
                        std::string(#call) + ": " + cudaGetErrorString(e__) + " (" + __FILE__ + ":" + std::to_string(__LINE__) + ")"); \
    } while (0)

template <typename T> int dev_alloc(kzgpu_ctx *ctx, DevMem &m, size_t count, T **out) {
    KZ_CUDA(ctx, m.alloc(count * sizeof(T)));
    *out = m.as<T>();
    return KZ_OK;
}
template <typename T> int dev_upload(kzgpu_ctx *ctx, Device &d, DevMem &m, const T *src, size_t count, const T **out) {
    T *p = nullptr;
    int rc = dev_alloc(ctx, m, count, &p);
    if (rc) return rc;
    if (count) KZ_CUDA(ctx, cudaMemcpyAsync(p, src, count * sizeof(T), cudaMemcpyHostToDevice, d.stream));
    *out = p;
    return KZ_OK;
}
/* Short-lived buffers (ingest staging, the builders' triangle list) come from the device's stream-ordered memory pool: a plain
 * cudaMalloc maps every new block into all peers once peer access is enabled (multi-device contexts, NCCL in the same process). */
template <typename T> int temp_alloc(kzgpu_ctx *ctx, AsyncMem &m, size_t count, cudaStream_t s, T **out) {
    KZ_CUDA(ctx, m.alloc(count * sizeof(T), s));
    *out = m.as<T>();
    return KZ_OK;
}
const size_t SCRATCH_MIN = 1u << 20;     /* the scratch buffers of the host-pointer entry points never shrink, nor start below this */

cudaEvent_t get_event(Device &d) {
    if (!d.free_events.empty()) { cudaEvent_t e = d.free_events.back(); d.free_events.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    if (cudaEventCreate(&e) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return e;
}
struct Timed {   /* records an event pair around a group of launches on `s`; timing is dropped (never the work) if events run out */
    Device &d; cudaStream_t s; EvPair p; bool ok;
    Timed(Device &dev, cudaStream_t st, int cat) : d(dev), s(st) {
        p.a = get_event(d); p.b = get_event(d); p.cat = cat;
        ok = p.a && p.b && cudaEventRecord(p.a, s) == cudaSuccess;
    }
    ~Timed() {
        if (ok && cudaEventRecord(p.b, s) == cudaSuccess) { d.pending.push_back(p); return; }
        if (p.a) d.free_events.push_back(p.a);
        if (p.b) d.free_events.push_back(p.b);
    }
};
/* Folds finished event pairs into the per-category totals (synchronises on them). */
void fold_events(Device &d) {
    for (EvPair &p : d.pending) {
        cudaEventSynchronize(p.b);
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) d.ms[p.cat] += ms;
        d.free_events.push_back(p.a); d.free_events.push_back(p.b);
    }
    d.pending.clear();
}

template <typename K> int persistent_grid(const Device &d, K kernel, int threads) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
    return d.sm_count * per_sm;
}

int select(kzgpu_ctx *ctx, int device, Device **out) {
    if (!ctx) return fail(nullptr, KZ_ERR_INVALID, "null context");
    if (device < 0 || device >= (int)ctx->devs.size()) return fail(ctx, KZ_ERR_INVALID, "device index out of range");
    Device &d = ctx->devs[(size_t)device];
    KZ_CUDA(ctx, cudaSetDevice(d.id));
    *out = &d;
    return KZ_OK;
}

bool is_device_ptr(const void *p) {
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeDevice;
}

int grid_for(size_t n, int threads, int sm_count) {
    const size_t blocks = (n + (size_t)threads - 1) / (size_t)threads;
    return (int)std::max<size_t>(1, std::min<size_t>(blocks, (size_t)sm_count * 16));
}

/* Small tables + frame of one device; the bulk arrays (vertex / index records, texels) are filled by ingest_geometry on the
 * first device and copied to the others over NVLink (replicate_geometry). */
int upload_tables(kzgpu_ctx *ctx, Device &d) {
    const KzHostScene &h = *ctx->hs;
    d.tables.clear();
    d.frame_mem.reset();
    d.sc = h.sc;     /* flatten() without geometry leaves the accel fields of h.sc empty, as drop_all() left those of d.sc */
    auto next = [&d]() -> DevMem & { d.tables.emplace_back(); return d.tables.back(); };
    int rc;
#define UP(field, vec) if ((rc = dev_upload(ctx, d, next(), (vec).data(), (vec).size(), &d.sc.field))) return rc
    UP(meshes, h.meshes);
    UP(light_cdf, h.light_cdf); UP(light_meshes, h.light_meshes); UP(bsdfs, h.bsdfs); UP(textures, h.textures);
    UP(images, h.images); UP(lights, h.lights); UP(blue_noise, h.blue_noise); UP(pmj02bn, h.pmj);
    UP(pmj_pixel_samples, h.pmj_pixel_samples);
#undef UP
    KzVertex *v = nullptr; KzU4 *ix = nullptr; KzF4 *tx = nullptr;
    if ((rc = dev_alloc(ctx, next(), (size_t)h.total_vertices, &v))) return rc;
    if ((rc = dev_alloc(ctx, next(), (size_t)h.total_triangles, &ix))) return rc;
    if ((rc = dev_alloc(ctx, next(), h.total_texels, &tx))) return rc;
    d.sc.vertices = v; d.sc.indices = ix; d.sc.texels = tx;
    /* frame */
    const size_t texels = (size_t)(h.sc.camera.width + 2 * h.sc.border) * (size_t)(h.sc.camera.height + 2 * h.sc.border);
    if ((rc = dev_alloc(ctx, d.frame_mem, texels, &d.frame))) return rc;
    d.frame_texels = texels;
    KZ_CUDA(ctx, cudaMemsetAsync(d.frame, 0, texels * sizeof(KzF4), d.stream));
    return KZ_OK;
}

/* Mesh and image arrays -> HBM records on device `d` (kz_ingest.cuh).  Host arrays are copied into a staging buffer with one
 * cudaMemcpyAsync each; arrays that already live on a device are read where they are. */
int ingest_geometry(kzgpu_ctx *ctx, Device &d, const kz_scene_desc *scene) {
    const KzHostScene &h = *ctx->hs;
    size_t stage_bytes = 0;
    for (uint32_t g = 0; g < scene->n_meshes; ++g) {
        const kz_mesh_desc &m = scene->meshes[g];
        stage_bytes = std::max(stage_bytes, (size_t)m.n_vertices * 32 + (size_t)m.n_triangles * 12 + 64);
    }
    for (uint32_t i = 0; i < scene->n_images; ++i) stage_bytes = std::max(stage_bytes, (size_t)scene->images[i].width * scene->images[i].height * 12);
    AsyncMem stage_mem, bad_mem;
    char *stage = nullptr; uint32_t *bad = nullptr;
    int rc;
    if ((rc = temp_alloc(ctx, stage_mem, stage_bytes, d.stream, &stage))) return rc;
    if ((rc = temp_alloc(ctx, bad_mem, 4, d.stream, &bad))) return rc;
    cudaError_t e = cudaMemsetAsync(bad, 0, 4, d.stream);
    auto fetch = [&](const void *src, size_t bytes, size_t &cursor) -> const void * {      /* device-visible view of a caller array */
        if (!src || e != cudaSuccess) return nullptr;
        if (is_device_ptr(src)) return src;
        char *dst = stage + cursor;
        cursor += (bytes + 15) & ~(size_t)15;
        e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, d.stream);
        return dst;
    };
    KzVertex *vertices = const_cast<KzVertex *>(d.sc.vertices);
    KzU4 *indices = const_cast<KzU4 *>(d.sc.indices);
    KzF4 *texels = const_cast<KzF4 *>(d.sc.texels);
    for (uint32_t g = 0; g < scene->n_meshes && e == cudaSuccess; ++g) {
        const kz_mesh_desc &m = scene->meshes[g];
        const KzMeshRec &r = h.meshes[g];
        size_t cur = 0;
        const float *pos = (const float *)fetch(m.positions, (size_t)m.n_vertices * 12, cur);
        const float *nrm = (const float *)fetch(m.normals, (size_t)m.n_vertices * 12, cur);
        const float *uv = (const float *)fetch(m.uvs, (size_t)m.n_vertices * 8, cur);
        const uint32_t *idx = (const uint32_t *)fetch(m.indices, (size_t)m.n_triangles * 12, cur);
        if (e != cudaSuccess) break;
        if (m.n_vertices) { k_ingest_vertices<<<grid_for(m.n_vertices, 256, d.sm_count), 256, 0, d.stream>>>(pos, nrm, uv, m.n_vertices, vertices + r.vertex_offset); ++d.launches; }
        if (m.n_triangles) { k_ingest_indices<<<grid_for(m.n_triangles, 256, d.sm_count), 256, 0, d.stream>>>(idx, m.n_triangles, m.n_vertices, indices + r.index_offset, bad); ++d.launches; }
    }
    for (uint32_t i = 0; i < scene->n_images && e == cudaSuccess; ++i) {
        const kz_image_desc &im = scene->images[i];
        const size_t n = (size_t)im.width * im.height;
        size_t cur = 0;
        const float *rgb = (const float *)fetch(im.rgb, n * 12, cur);
        if (e != cudaSuccess) break;
        k_ingest_texels<<<grid_for(n, 256, d.sm_count), 256, 0, d.stream>>>(rgb, n, texels + h.images[i].texel_offset);
        ++d.launches;
    }
    uint32_t h_bad = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h_bad, bad, 4, cudaMemcpyDeviceToHost, d.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(d.stream);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, KZ_ERR_CUDA, std::string("scene ingest: ") + cudaGetErrorString(e));
    if (h_bad) return fail(ctx, KZ_ERR_INVALID, "vertex index out of range");
    return KZ_OK;
}

/* Copies the ingested records of `src` into the (already allocated) arrays of `dst`: peer copies over NVLink. */
int replicate_geometry(kzgpu_ctx *ctx, Device &dst, const Device &src) {
    const KzHostScene &h = *ctx->hs;
    KZ_CUDA(ctx, cudaMemcpyPeerAsync(const_cast<KzVertex *>(dst.sc.vertices), dst.id, src.sc.vertices, src.id, (size_t)h.total_vertices * sizeof(KzVertex), dst.stream));
    KZ_CUDA(ctx, cudaMemcpyPeerAsync(const_cast<KzU4 *>(dst.sc.indices), dst.id, src.sc.indices, src.id, (size_t)h.total_triangles * sizeof(KzU4), dst.stream));
    KZ_CUDA(ctx, cudaMemcpyPeerAsync(const_cast<KzF4 *>(dst.sc.texels), dst.id, src.sc.texels, src.id, h.total_texels * sizeof(KzF4), dst.stream));
    KZ_CUDA(ctx, cudaStreamSynchronize(dst.stream));
    return KZ_OK;
}

int ensure_pool(kzgpu_ctx *ctx, Lane &L, uint32_t cap) {
    if (L.pool_cap >= cap) return KZ_OK;
    for (DevMem &m : L.pool) m.reset();     /* the old pool goes before the new one is allocated */
    L.pool_cap = 0;
    DevMem *m = L.pool;
    int rc;
#define AL(ptr) if ((rc = dev_alloc(ctx, *m++, (size_t)cap, &(ptr)))) return rc
    AL(L.st.a); AL(L.st.b); AL(L.st.c);
    AL(L.q.ext[0]); AL(L.q.ext[1]); AL(L.q.shadow);
    for (int c = 0; c < KZ_NUM_CLASSES; ++c) AL(L.q.cls[c]);
#undef AL
    L.pool_cap = cap;
    return KZ_OK;
}

/* install() and drop_all() are the only places where the accel of a device changes.  drop_all() releases the accel of every
 * device and clears ctx->built, which only a completed build or refit sets again: from the moment an old accel is released until a
 * new one is installed on every device, trace and render return KZ_ERR_STATE instead of reading released memory. */
void install(Device &d, Accel &&a) {
    d.accel = std::move(a);
    d.sc.nodes = d.accel.nodes.as<const KzNode8>(); d.sc.tris = d.accel.tris.as<const KzF4>();
    d.sc.n_nodes = d.accel.n_nodes; d.sc.n_tris = d.accel.n_tris; d.sc.scene_max_abs = d.accel.max_abs;
    d.has_accel = true;
    d.hint_stale = true;
    d.levels_checked = false;
}
void drop_all(kzgpu_ctx *ctx) {
    ctx->built = false;
    ctx->levels.clear();
    for (Device &d : ctx->devs) {
        cudaSetDevice(d.id);
        d.accel = Accel();
        d.sc.nodes = nullptr; d.sc.tris = nullptr; d.sc.n_nodes = 0; d.sc.n_tris = 0; d.sc.scene_max_abs = 0.f;
        d.has_accel = false;
    }
}

int upload_accel(kzgpu_ctx *ctx, Device &d, const kzbvh::Built &b) {
    Accel a{{}, {}, (uint32_t)b.nodes.size(), (uint32_t)(b.tris.size() / 3), b.max_abs};
    const KzNode8 *nodes; const KzF4 *tris;
    int rc;
    if ((rc = dev_upload(ctx, d, a.nodes, b.nodes.data(), b.nodes.size(), &nodes))) return rc;
    if ((rc = dev_upload(ctx, d, a.tris, b.tris.data(), b.tris.size(), &tris))) return rc;
    KZ_CUDA(ctx, cudaStreamSynchronize(d.stream));
    install(d, std::move(a));
    return KZ_OK;
}

/* Copies the accel of device `src` into fresh arrays of `dst` (current; peer copies over NVLink). */
int replicate_accel(kzgpu_ctx *ctx, Device &dst, const Device &src) {
    Accel a{{}, {}, src.accel.n_nodes, src.accel.n_tris, src.accel.max_abs};
    KzNode8 *nodes = nullptr; KzF4 *tris = nullptr;
    int rc;
    if ((rc = dev_alloc(ctx, a.nodes, (size_t)a.n_nodes, &nodes))) return rc;
    if ((rc = dev_alloc(ctx, a.tris, (size_t)a.n_tris * 3, &tris))) return rc;
    KZ_CUDA(ctx, cudaMemcpyPeerAsync(nodes, dst.id, src.sc.nodes, src.id, (size_t)a.n_nodes * sizeof(KzNode8), dst.stream));
    KZ_CUDA(ctx, cudaMemcpyPeerAsync(tris, dst.id, src.sc.tris, src.id, (size_t)a.n_tris * 3 * sizeof(KzF4), dst.stream));
    KZ_CUDA(ctx, cudaStreamSynchronize(dst.stream));
    install(dst, std::move(a));
    return KZ_OK;
}

/* One chunk of path slots through the whole wavefront on stream `s` with the pool of lane `L`; never synchronises (except the
 * unbounded whitted / path_mats loops, which poll a queue count). */
/* `ectx` receives error messages (nullptr inside the per-device worker threads of kzgpu_render, which report through g_error). */
#ifndef KZ_HINT_MIN_TRIS
#define KZ_HINT_MIN_TRIS (1u << 20)
#endif
bool hints_on(const kzgpu_ctx *ctx) {
    return ctx->primary_hint == 2 || (ctx->primary_hint == 1 && ctx->hs->total_triangles >= KZ_HINT_MIN_TRIS);
}

int enqueue_chunk(const kzgpu_ctx *ctx, kzgpu_ctx *ectx, Device &d, Lane &L, const KzChunk &ch, unsigned long long new_paths, cudaStream_t s) {
    const KzScene &sc = d.sc;
    const int max_depth = sc.integrator.max_depth;
    /* the pass after the last vertex only resolves "miss -> background" (integrator.cpp:315-318) */
    const int last_pass = sc.background >= 0 ? max_depth : max_depth - 1;
    const bool alt = sc.integrator.type != KZ_INTEGRATOR_PATH_MIS;
    uint2 *const hint = hints_on(ctx) ? d.hint.as<uint2>() : nullptr;
    if (d.pending.size() > 8192) fold_events(d);       /* very long renders: bound the number of live timing events */
    {
        Timed t(d, s, CAT_SHADE);
        k_chunk_reset<<<1, 32, 0, s>>>(L.ctl, ch.count, new_paths);
        k_raygen<<<(ch.count + KZ_SHADE_THREADS - 1) / KZ_SHADE_THREADS, KZ_SHADE_THREADS, 0, s>>>(sc, L.st, hint, ch);
        d.launches += 2;
    }
    if (alt) {
        /* normals / ao: one pass; whitted / path_mats: unbounded loops ended by Russian roulette -- the only place the host
         * looks at a queue count (every 8 passes), because these loops have no a-priori length */
        const int passes = (sc.integrator.type == KZ_INTEGRATOR_NORMALS || sc.integrator.type == KZ_INTEGRATOR_AO) ? 1 : 4096;
        for (int b = 0; b < passes; ++b) {
            const int cur = b & 1, nxt = cur ^ 1;
            {
                Timed t(d, s, CAT_TRACE);
                k_bounce_reset<<<1, 32, 0, s>>>(L.ctl, nxt);
                if (b == 0) k_extend<true><<<d.grid_extend0, KZ_TRACE_THREADS, 0, s>>>(sc, L.st, L.ctl, L.q, cur, hint);
                else k_extend<false><<<d.grid_extend, KZ_TRACE_THREADS, 0, s>>>(sc, L.st, L.ctl, L.q, cur, nullptr);
                d.launches += 2;
            }
            {
                Timed t(d, s, CAT_SHADE);
                k_shade<KZ_CLASS_GENERIC><<<d.grid_shade[4], KZ_SHADE_THREADS, 0, s>>>(sc, L.st, L.ctl, L.q, nxt, b);
                ++d.launches;
            }
            if (sc.integrator.type == KZ_INTEGRATOR_AO || sc.integrator.type == KZ_INTEGRATOR_WHITTED) {
                Timed t(d, s, CAT_TRACE);
                k_shadow<<<d.grid_shadow, KZ_TRACE_THREADS, 0, s>>>(sc, L.st, L.ctl, L.q, nxt);
                ++d.launches;
            }
            if (passes > 1 && (b & 7) == 7) {
                unsigned long long left = 0;
                KZ_CUDA(ectx, cudaMemcpyAsync(&left, &L.ctl->ext_shadow[nxt], sizeof(left), cudaMemcpyDeviceToHost, s));
                KZ_CUDA(ectx, cudaStreamSynchronize(s));
                if ((left & 0xFFFFFFFFull) == 0ull) break;
            }
        }
    } else
    for (int b = 0; b <= last_pass; ++b) {
        const int cur = b & 1, nxt = cur ^ 1;
        {
            Timed t(d, s, CAT_TRACE);
            k_bounce_reset<<<1, 32, 0, s>>>(L.ctl, nxt);
            if (b == 0) k_extend<true><<<d.grid_extend0, KZ_TRACE_THREADS, 0, s>>>(sc, L.st, L.ctl, L.q, cur, hint);
            else k_extend<false><<<d.grid_extend, KZ_TRACE_THREADS, 0, s>>>(sc, L.st, L.ctl, L.q, cur, nullptr);
            d.launches += 2;
        }
        {
            Timed t(d, s, CAT_SHADE);
            k_shade<KZ_CLASS_TERMINAL><<<d.grid_shade[0], KZ_SHADE_THREADS, 0, s>>>(sc, L.st, L.ctl, L.q, nxt, b);
            ++d.launches;
            if (b < max_depth) {
                if (ctx->class_present[KZ_CLASS_DIFFUSE]) { k_shade<KZ_CLASS_DIFFUSE><<<d.grid_shade[1], KZ_SHADE_THREADS, 0, s>>>(sc, L.st, L.ctl, L.q, nxt, b); ++d.launches; }
                if (ctx->class_present[KZ_CLASS_KISS]) { k_shade<KZ_CLASS_KISS><<<d.grid_shade[2], KZ_SHADE_THREADS, 0, s>>>(sc, L.st, L.ctl, L.q, nxt, b); ++d.launches; }
                if (ctx->class_present[KZ_CLASS_NORMALMAP]) { k_shade<KZ_CLASS_NORMALMAP><<<d.grid_shade[3], KZ_SHADE_THREADS, 0, s>>>(sc, L.st, L.ctl, L.q, nxt, b); ++d.launches; }
                if (ctx->class_present[KZ_CLASS_GENERIC]) { k_shade<KZ_CLASS_GENERIC><<<d.grid_shade[4], KZ_SHADE_THREADS, 0, s>>>(sc, L.st, L.ctl, L.q, nxt, b); ++d.launches; }
            }
        }
        if (b < max_depth && sc.n_light_meshes > 0) {
            Timed t(d, s, CAT_TRACE);
            k_shadow<<<d.grid_shadow, KZ_TRACE_THREADS, 0, s>>>(sc, L.st, L.ctl, L.q, nxt);
            ++d.launches;
        }
    }
    {
        Timed t(d, s, CAT_SHADE);
        /* (an earlier tiled variant pre-summed the taps of 256 neighbouring paths with shared-memory float atomics -- compare-and-swap
         * loops -- and was 10 % slower end to end; k_accumulate now sums a tile's sample indices conflict-free, see there) */
        k_accumulate<<<std::min<uint32_t>((ch.count + KZ_SHADE_THREADS - 1) / KZ_SHADE_THREADS, (uint32_t)d.sm_count * 16u), KZ_SHADE_THREADS, 0, s>>>(sc, L.st, ch.count, d.frame, ch.x0, ch.y0);
        ++d.launches;
    }
    return KZ_OK;
}

/* Enqueues the whole wavefront for one request; work is ordered after everything already on `s`, and `s` waits for it. */
int enqueue_render(const kzgpu_ctx *ctx, kzgpu_ctx *ectx, Device &d, const kz_render_req &req, cudaStream_t s) {
    const KzScene &sc = d.sc;
    const int w = req.x1 - req.x0, h = req.y1 - req.y0, nS = req.spp_end - req.spp_begin;
    if (w <= 0 || h <= 0 || nS <= 0) return KZ_OK;
    KzChunk ch;
    ch.x0 = req.x0; ch.y0 = req.y0; ch.x1 = req.x1; ch.y1 = req.y1;
    ch.tiles_x = (uint32_t)(w + 7) / 8u;
    const uint32_t tiles_y = (uint32_t)(h + 3) / 4u;
    ch.npx_padded = ch.tiles_x * tiles_y * 32u;
    ch.spp_begin = req.spp_begin;
    ch.n_spp = (uint32_t)nS;
    ch.spp_group = (uint32_t)std::min(nS, ctx->spp_group);
    const unsigned long long total = (unsigned long long)ch.npx_padded * (unsigned long long)nS;
    /* two lanes once there is enough work for two chunks (the unbounded loops of whitted / path_mats poll the host: one lane) */
    const bool alt = sc.integrator.type != KZ_INTEGRATOR_PATH_MIS;
    /* measured on B200 (Mpaths/s, pool 2^23 x 2 lanes -> 2^24 x 3): 10^8-triangle 4K headline 848 -> 866, configs[2] 826 -> 840, configs[3] 792 -> 812;
     * a 2^24-path frame (WarmStudio.xml 512x512x64) is best left on two lanes (1213 vs 1203) */
    const int lanes = (alt || total < (1ull << 21)) ? 1 : (total >= (1ull << 25) ? ctx->lanes : std::min(ctx->lanes, 2));
    /* equal chunks, a multiple of the lane count of them, none larger than the pool: the lanes finish together (4 chunks on 3 lanes
     * would leave two lanes idle for the last quarter of the frame) */
    const unsigned long long rounds = (total + (unsigned long long)lanes * ctx->pool_cap - 1) / ((unsigned long long)lanes * ctx->pool_cap);
    const unsigned long long n_chunks = rounds * (unsigned long long)lanes;
    const uint32_t cap = (uint32_t)((((total + n_chunks - 1) / n_chunks) + 31ull) & ~31ull);
    int rc;
    for (int l = 0; l < lanes; ++l) if ((rc = ensure_pool(ectx, d.lane[l], cap))) return rc;
    if (hints_on(ctx)) {
        /* every pixel k_raygen can produce lies on the film (check_req), whatever the rectangle or the device's share of samples */
        const size_t bytes = (size_t)sc.camera.width * (size_t)sc.camera.height * sizeof(uint2);
        if (d.hint.bytes < bytes) {
            KZ_CUDA(ectx, d.hint.alloc(bytes));
            d.hint_stale = true;
        }
        if (d.hint_stale) {     /* before anything of this request, on s: the other lanes start after it (below) */
            KZ_CUDA(ectx, cudaMemsetAsync(d.hint.p, 0xFF, d.hint.bytes, s));
            d.hint_stale = false;
        }
    }
    Timed total_t(d, s, CAT_TOTAL);
    if (lanes > 1) {       /* the other lanes start after what is already queued on s (frame clear, earlier requests) */
        KZ_CUDA(ectx, cudaEventRecord(d.lane[0].done, s));
        for (int l = 1; l < lanes; ++l) KZ_CUDA(ectx, cudaStreamWaitEvent(d.lane[l].stream, d.lane[0].done, 0));
    }
    int k = 0;
    for (unsigned long long first = 0; first < total; first += cap, ++k) {
        Lane &L = d.lane[k % lanes];
        ch.first = first;
        ch.count = (uint32_t)std::min<unsigned long long>(cap, total - first);
        const unsigned long long new_paths = first == 0 ? (unsigned long long)w * (unsigned long long)h * (unsigned long long)nS : 0ull;
        if ((rc = enqueue_chunk(ctx, ectx, d, L, ch, new_paths, (k % lanes) == 0 ? s : L.stream))) return rc;
    }
    for (int l = 1; l < lanes; ++l) {
        KZ_CUDA(ectx, cudaEventRecord(d.lane[l].done, d.lane[l].stream));
        KZ_CUDA(ectx, cudaStreamWaitEvent(s, d.lane[l].done, 0));
    }
    KZ_CUDA(ectx, cudaGetLastError());
    return KZ_OK;
}

int check_ready(kzgpu_ctx *ctx, bool need_accel) {
    if (!ctx) return fail(nullptr, KZ_ERR_INVALID, "null context");
    if (!ctx->uploaded) return fail(ctx, KZ_ERR_STATE, "no scene uploaded");
    if (need_accel && !ctx->built)
        return fail(ctx, KZ_ERR_STATE, ctx->devs[0].has_accel ? "the vertices changed since the accel was built: call kzgpu_accel_refit or kzgpu_accel_build"
                                                              : "accel not built: call kzgpu_accel_build first");
    return KZ_OK;
}

}  // namespace

extern "C" {

const char *kzgpu_last_error(const kzgpu_ctx *ctx) { return ctx ? ctx->error.c_str() : g_error.c_str(); }

int kzgpu_create(const int *device_ids, int n_devices, kzgpu_ctx **out) {
    if (!out) return fail(nullptr, KZ_ERR_INVALID, "null out pointer");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(nullptr, KZ_ERR_NO_DEVICE, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                                                    " (kzgpu has no CPU fallback)");
    std::vector<int> ids;
    if (!device_ids || n_devices <= 0) ids.push_back(0);
    else ids.assign(device_ids, device_ids + n_devices);
    std::unique_ptr<kzgpu_ctx> ctx(new kzgpu_ctx());
    if (const char *p = getenv("KZGPU_POOL_LOG2")) { int l = atoi(p); if (l >= 10 && l <= 26) ctx->pool_cap = 1u << l; }
    if (const char *p = getenv("KZGPU_LANES")) { int l = atoi(p); if (l >= 1 && l <= KZ_MAX_LANES) ctx->lanes = l; }
    if (const char *p = getenv("KZGPU_SPP_GROUP")) { int g = atoi(p); if (g >= 1) ctx->spp_group = g; }
    if (const char *p = getenv("KZGPU_PRIMARY_HINT")) { int h = atoi(p); if (h >= 0 && h <= 2) ctx->primary_hint = h; }
    /* the devices are set up in place and never move (code compares &d with &ctx->devs[0]); a failure below releases all of them */
    ctx->devs = std::vector<Device>(ids.size());
    for (size_t i = 0; i < ids.size(); ++i) {
        const int id = ids[i];
        if (id < 0 || id >= count) return fail(nullptr, KZ_ERR_NO_DEVICE, "device id " + std::to_string(id) + " out of range");
        cudaDeviceProp prop;
        KZ_CUDA(nullptr, cudaGetDeviceProperties(&prop, id));
        if (prop.major != 10) return fail(nullptr, KZ_ERR_NO_DEVICE, std::string("device ") + prop.name + " is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                                                                       "; this library is built for sm_100a only");
        KZ_CUDA(nullptr, cudaSetDevice(id));
        Device &d = ctx->devs[i];
        d.id = id; d.sm_count = prop.multiProcessorCount;
        KZ_CUDA(nullptr, cudaStreamCreateWithFlags(&d.stream.h, cudaStreamNonBlocking));
        for (Lane &L : d.lane) {
            KZ_CUDA(nullptr, L.ctl_mem.alloc(sizeof(KzControl)));
            L.ctl = L.ctl_mem.as<KzControl>();
            KZ_CUDA(nullptr, cudaMemset(L.ctl, 0, sizeof(KzControl)));
            KZ_CUDA(nullptr, cudaEventCreateWithFlags(&L.done.h, cudaEventDisableTiming));
        }
        for (int l = 1; l < KZ_MAX_LANES; ++l) KZ_CUDA(nullptr, cudaStreamCreateWithFlags(&d.lane[l].stream.h, cudaStreamNonBlocking));
        d.ctl = d.lane[0].ctl;
        KZ_CUDA(nullptr, cudaEventCreateWithFlags(&d.splat_done.h, cudaEventDisableTiming));
        KZ_CUDA(nullptr, cudaEventCreateWithFlags(&d.merge_done.h, cudaEventDisableTiming));
        KZ_CUDA(nullptr, d.cursor.alloc(64));
        d.grid_extend0 = persistent_grid(d, k_extend<true>, KZ_TRACE_THREADS);
        d.grid_extend = persistent_grid(d, k_extend<false>, KZ_TRACE_THREADS);
        d.grid_shadow = persistent_grid(d, k_shadow, KZ_TRACE_THREADS);
        d.grid_trace = persistent_grid(d, k_trace, KZ_TRACE_THREADS);
        if (const char *p = getenv("KZGPU_TRACE_CTAS_PER_SM")) { const int k = atoi(p); if (k >= 1 && k <= 16) d.grid_trace = d.sm_count * k; }     /* tuning experiments */
        d.grid_occ = persistent_grid(d, k_occluded, KZ_TRACE_THREADS);
        d.grid_shade[0] = persistent_grid(d, k_shade<KZ_CLASS_TERMINAL>, KZ_SHADE_THREADS);
        d.grid_shade[1] = persistent_grid(d, k_shade<KZ_CLASS_DIFFUSE>, KZ_SHADE_THREADS);
        d.grid_shade[2] = persistent_grid(d, k_shade<KZ_CLASS_KISS>, KZ_SHADE_THREADS);
        d.grid_shade[3] = persistent_grid(d, k_shade<KZ_CLASS_NORMALMAP>, KZ_SHADE_THREADS);
        d.grid_shade[4] = persistent_grid(d, k_shade<KZ_CLASS_GENERIC>, KZ_SHADE_THREADS);
    }
    /* a multi-device context replicates the scene and merges the frames through peer memory (NVLink / NVSwitch): every pair of its
     * devices must be able to map each other's HBM */
    if (ctx->devs.size() > KZ_MAX_DEVICES) return fail(nullptr, KZ_ERR_INVALID, "more than " + std::to_string(KZ_MAX_DEVICES) + " devices in one context");
    for (const Device &a : ctx->devs)
        for (const Device &b : ctx->devs) {
            if (a.id == b.id) { if (&a != &b) return fail(nullptr, KZ_ERR_INVALID, "device listed twice"); continue; }
            int ok = 0;
            KZ_CUDA(nullptr, cudaDeviceCanAccessPeer(&ok, a.id, b.id));
            if (!ok) return fail(nullptr, KZ_ERR_UNSUPPORTED, "devices " + std::to_string(a.id) + " and " + std::to_string(b.id) + " have no peer access; multi-device contexts need NVLink/PCIe P2P");
            KZ_CUDA(nullptr, cudaSetDevice(a.id));
            const cudaError_t e = cudaDeviceEnablePeerAccess(b.id, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
            else KZ_CUDA(nullptr, e);
        }
    *out = ctx.release();
    return KZ_OK;
}

void kzgpu_destroy(kzgpu_ctx *ctx) {
    if (!ctx) return;
    for (Device &d : ctx->devs) {
        cudaSetDevice(d.id);
        fold_events(d);
    }
    delete ctx;     /* ~Device synchronises each device and releases its resources */
}

int kzgpu_scene_upload(kzgpu_ctx *ctx, const kz_scene_desc *scene) {
    if (!ctx) return fail(nullptr, KZ_ERR_INVALID, "null context");
    if (!scene) return fail(ctx, KZ_ERR_INVALID, "null scene");
    const auto t0 = std::chrono::steady_clock::now();
    /* emitters need their positions / indices on the host for the area CDF (Mesh::activate, mesh.cpp:24-45): if such a mesh was
     * handed over as device arrays, read them back (emitters are small) */
    std::vector<kz_mesh_desc> meshes(scene->meshes, scene->meshes + (scene->meshes ? scene->n_meshes : 0));
    std::vector<std::vector<float>> host_pos; std::vector<std::vector<uint32_t>> host_idx;
    for (kz_mesh_desc &m : meshes) {
        if (m.light < 0 || !m.positions || !m.indices) continue;
        if (is_device_ptr(m.positions)) {
            host_pos.emplace_back((size_t)m.n_vertices * 3);
            KZ_CUDA(ctx, cudaMemcpy(host_pos.back().data(), m.positions, (size_t)m.n_vertices * 12, cudaMemcpyDeviceToHost));
            m.positions = host_pos.back().data();
        }
        if (is_device_ptr(m.indices)) {
            host_idx.emplace_back((size_t)m.n_triangles * 3);
            KZ_CUDA(ctx, cudaMemcpy(host_idx.back().data(), m.indices, (size_t)m.n_triangles * 12, cudaMemcpyDeviceToHost));
            m.indices = host_idx.back().data();
        }
    }
    kz_scene_desc tables = *scene;
    tables.meshes = meshes.data();
    std::unique_ptr<KzHostScene> hs(new KzHostScene());
    if (!hs->flatten(&tables, /*geometry=*/false)) {
        const bool unsupported = hs->error.find("outside the hot-path scope") != std::string::npos || hs->error.find("unsupported") != std::string::npos;
        return fail(ctx, unsupported ? KZ_ERR_UNSUPPORTED : KZ_ERR_INVALID, hs->error);
    }
    ctx->hs = std::move(hs);
    ctx->uploaded = false;
    drop_all(ctx);
    for (int c = 1; c < KZ_NUM_CLASSES; ++c) ctx->class_present[c] = false;
    for (const KzMeshRec &m : ctx->hs->meshes) {
        if (m.flags & KZ_MESH_IS_LIGHT) continue;
        const int t = ctx->hs->bsdfs[(size_t)m.bsdf].type;
        ctx->class_present[t == KZ_BSDF_DIFFUSE ? KZ_CLASS_DIFFUSE : (t == KZ_BSDF_KISS ? KZ_CLASS_KISS : (t == KZ_BSDF_NORMALMAP ? KZ_CLASS_NORMALMAP : KZ_CLASS_GENERIC))] = true;
    }
    for (Device &d : ctx->devs) {
        KZ_CUDA(ctx, cudaSetDevice(d.id));
        int rc = upload_tables(ctx, d);
        if (rc) return rc;
        /* the first device ingests the caller's arrays, the others get its records over NVLink */
        if (&d == &ctx->devs[0]) rc = ingest_geometry(ctx, d, scene);
        else rc = replicate_geometry(ctx, d, ctx->devs[0]);
        if (rc) return rc;
    }
    KZ_CUDA(ctx, cudaSetDevice(ctx->devs[0].id));
    ctx->uploaded = true;
    ctx->ms_upload = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return KZ_OK;
}

int kzgpu_accel_build(kzgpu_ctx *ctx, int builder) {
    int rc = check_ready(ctx, false);
    if (rc) return rc;
    if (builder != KZ_BUILD_HOST_SAH && builder != KZ_BUILD_LBVH) return fail(ctx, KZ_ERR_INVALID, "unknown builder");
    const auto t0 = std::chrono::steady_clock::now();
    Device &d0 = ctx->devs[0];
    KZ_CUDA(ctx, cudaSetDevice(d0.id));
    /* the builders' input: the triangle list in scene order, gathered on the device from the ingested records */
    const uint32_t n_tris = (uint32_t)ctx->hs->total_triangles;
    std::vector<uint32_t> levels;     /* -> ctx->levels once the new accel is installed everywhere */
    AsyncMem tris_mem;
    kzbvh::Tri *d_tris = nullptr;
    if ((rc = temp_alloc(ctx, tris_mem, (size_t)n_tris, d0.stream, &d_tris))) return rc;
    if (n_tris) {
        k_gather_tris<<<grid_for(n_tris, 256, d0.sm_count), 256, 0, d0.stream>>>(d0.sc.meshes, d0.sc.n_meshes, d0.sc.vertices, d0.sc.indices, n_tris, d_tris);
        ++d0.launches;
    }
    if (builder == KZ_BUILD_HOST_SAH) {
        std::vector<kzbvh::Tri> tris((size_t)n_tris);
        cudaError_t e = cudaSuccess;
        if (n_tris) e = cudaMemcpyAsync(tris.data(), d_tris, (size_t)n_tris * sizeof(kzbvh::Tri), cudaMemcpyDeviceToHost, d0.stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(d0.stream);
        tris_mem.reset();
        KZ_CUDA(ctx, e);
        kzbvh::Built built;
        kzbvh::buildHostSah(tris, 0, built);
        /* a failure up to here keeps the old accel in use */
        if (built.depth > KZ_MAX_ACCEL_DEPTH) return fail(ctx, KZ_ERR_UNSUPPORTED, "accel deeper than the traversal stack allows");
        if (!kz_refit_levels(built.nodes.data(), (uint32_t)built.nodes.size(), levels)) levels.clear();
        drop_all(ctx);      /* the old accel goes before the new one is allocated: at 10^8 triangles one is about 13 GB */
        for (Device &d : ctx->devs) {
            KZ_CUDA(ctx, cudaSetDevice(d.id));
            if ((rc = upload_accel(ctx, d, built))) return rc;
        }
        ctx->bvh_nodes = built.nodes.size();
        ctx->bvh_bytes = built.nodes.size() * sizeof(KzNode8) + built.tris.size() * sizeof(KzF4);
    } else {
        drop_all(ctx);
        KZ_CUDA(ctx, cudaSetDevice(d0.id));
        kzlbvh::Result r;
        std::string err;
        rc = kzlbvh::build(d_tris, n_tris, d0.stream, r, err);
        tris_mem.reset();
        /* hand the pool's memory back: the path pools and the caller's own allocations need it, the next build allocates afresh */
        { cudaMemPool_t pool; if (cudaDeviceGetDefaultMemPool(&pool, d0.id) == cudaSuccess) { cudaStreamSynchronize(d0.stream); cudaMemPoolTrimTo(pool, 0); } }
        if (rc) return fail(ctx, rc, err);
        if (r.depth > KZ_MAX_ACCEL_DEPTH) return fail(ctx, KZ_ERR_UNSUPPORTED, "accel deeper than the traversal stack allows");
        install(d0, Accel{std::move(r.nodes), std::move(r.tris), r.n_nodes, r.n_tris, r.max_abs});
        levels = r.n_nodes ? r.level_first : std::vector<uint32_t>(1, 0u);
        if (levels.back() != r.n_nodes) levels.clear();
        d0.launches += r.launches;
        ctx->bvh_nodes = r.n_nodes;
        ctx->bvh_bytes = (uint64_t)r.n_nodes * sizeof(KzNode8) + (uint64_t)r.n_tris * 3 * sizeof(KzF4);
        /* built once; the other devices get the arrays over NVLink */
        for (size_t g = 1; g < ctx->devs.size(); ++g) {
            KZ_CUDA(ctx, cudaSetDevice(ctx->devs[g].id));
            if ((rc = replicate_accel(ctx, ctx->devs[g], d0))) return rc;
        }
        KZ_CUDA(ctx, cudaSetDevice(d0.id));
    }
    ctx->ms_build = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    ctx->levels = std::move(levels);
    ctx->built = true;
    return KZ_OK;
}

int kzgpu_mesh_update(kzgpu_ctx *ctx, int mesh, const float *positions, const float *normals) {
    if (!ctx) return fail(nullptr, KZ_ERR_INVALID, "null context");
    if (!ctx->uploaded) return fail(ctx, KZ_ERR_STATE, "no scene uploaded");
    KzHostScene &h = *ctx->hs;
    if (mesh < 0 || mesh >= (int)h.meshes.size()) return fail(ctx, KZ_ERR_INVALID, "mesh index out of range");
    if (!positions) return fail(ctx, KZ_ERR_INVALID, "null positions");
    KzMeshRec &r = h.meshes[(size_t)mesh];
    if (normals && !(r.flags & KZ_MESH_HAS_NORMALS)) return fail(ctx, KZ_ERR_INVALID, "normals given for a mesh uploaded without normals");
    const uint32_t nv = (uint32_t)(((size_t)mesh + 1 < h.meshes.size() ? (uint64_t)h.meshes[(size_t)mesh + 1].vertex_offset : h.total_vertices) - r.vertex_offset);
    Device &d0 = ctx->devs[0];
    KZ_CUDA(ctx, cudaSetDevice(d0.id));
    /* an emitter's area CDF, normalisation and bounds are recomputed on the host from its new positions (read back if they are a
     * device array, as kzgpu_scene_upload does) and its index records (read back from HBM); nothing is written before this succeeded */
    std::vector<float> cdf, bounds(6);
    float inv_area = 0.f;
    size_t light_k = 0;
    if (r.flags & KZ_MESH_IS_LIGHT) {
        std::vector<float> pos;
        const float *hp = positions;
        if (is_device_ptr(positions)) {
            pos.resize((size_t)nv * 3);
            KZ_CUDA(ctx, cudaMemcpy(pos.data(), positions, (size_t)nv * 12, cudaMemcpyDeviceToHost));
            hp = pos.data();
        }
        std::vector<KzU4> rec(r.n_triangles);
        KZ_CUDA(ctx, cudaMemcpyAsync(rec.data(), d0.sc.indices + r.index_offset, (size_t)r.n_triangles * sizeof(KzU4), cudaMemcpyDeviceToHost, d0.stream));
        KZ_CUDA(ctx, cudaStreamSynchronize(d0.stream));
        std::vector<uint32_t> idx((size_t)r.n_triangles * 3);
        for (size_t f = 0; f < rec.size(); ++f) { idx[3 * f] = rec[f].x; idx[3 * f + 1] = rec[f].y; idx[3 * f + 2] = rec[f].z; }
        cdf.resize((size_t)r.n_triangles + 1);
        KzHostScene::emitter_tables(hp, idx.data(), r.n_triangles, cdf.data(), inv_area, bounds.data());
        while (h.light_meshes[light_k] != mesh) ++light_k;
    }
    /* from here on the scene changes: the accel no longer matches it until a refit or a build */
    ctx->built = false;
    /* vertex records of device 0: host arrays are staged with one copy each, device arrays read in place */
    {
        AsyncMem stage_mem[2];
        const float *src[2] = {positions, normals};
        cudaError_t e = cudaSuccess;
        for (int k = 0; k < 2 && e == cudaSuccess; ++k) {
            if (!src[k] || is_device_ptr(src[k])) continue;
            float *stage = nullptr;
            int rc = temp_alloc(ctx, stage_mem[k], (size_t)nv * 3, d0.stream, &stage);
            if (rc) return rc;
            e = cudaMemcpyAsync(stage, src[k], (size_t)nv * 12, cudaMemcpyHostToDevice, d0.stream);
            src[k] = stage;
        }
        if (e == cudaSuccess && nv) {
            k_update_vertices<<<grid_for(nv, 256, d0.sm_count), 256, 0, d0.stream>>>(src[0], src[1], nv, const_cast<KzVertex *>(d0.sc.vertices) + r.vertex_offset);
            ++d0.launches;
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(d0.stream);
        if (e != cudaSuccess) return fail(ctx, KZ_ERR_CUDA, std::string("mesh update: ") + cudaGetErrorString(e));
    }
    if (r.flags & KZ_MESH_IS_LIGHT) {
        std::copy(cdf.begin(), cdf.end(), h.light_cdf.begin() + r.cdf_offset);
        r.inv_area = inv_area;
        std::copy(bounds.begin(), bounds.end(), h.light_bounds.begin() + 6 * light_k);
        h.invisible_light_bounds();
    }
    for (Device &d : ctx->devs) {
        KZ_CUDA(ctx, cudaSetDevice(d.id));
        if (&d != &d0 && nv)
            KZ_CUDA(ctx, cudaMemcpyPeerAsync(const_cast<KzVertex *>(d.sc.vertices) + r.vertex_offset, d.id, d0.sc.vertices + r.vertex_offset, d0.id, (size_t)nv * sizeof(KzVertex), d.stream));
        if (r.flags & KZ_MESH_IS_LIGHT) {
            KZ_CUDA(ctx, cudaMemcpyAsync(const_cast<KzMeshRec *>(d.sc.meshes), h.meshes.data(), h.meshes.size() * sizeof(KzMeshRec), cudaMemcpyHostToDevice, d.stream));
            KZ_CUDA(ctx, cudaMemcpyAsync(const_cast<float *>(d.sc.light_cdf), h.light_cdf.data(), h.light_cdf.size() * sizeof(float), cudaMemcpyHostToDevice, d.stream));
            for (int a = 0; a < 3; ++a) { d.sc.inv_light_lo[a] = h.sc.inv_light_lo[a]; d.sc.inv_light_hi[a] = h.sc.inv_light_hi[a]; }
        }
        KZ_CUDA(ctx, cudaStreamSynchronize(d.stream));
    }
    KZ_CUDA(ctx, cudaSetDevice(d0.id));
    return KZ_OK;
}

int kzgpu_accel_refit(kzgpu_ctx *ctx) {
    if (!ctx) return fail(nullptr, KZ_ERR_INVALID, "null context");
    if (!ctx->uploaded) return fail(ctx, KZ_ERR_STATE, "no scene uploaded");
    for (const Device &d : ctx->devs)
        if (!d.has_accel) return fail(ctx, KZ_ERR_STATE, "no accel built since the last upload: call kzgpu_accel_build first");
    if (ctx->levels.empty()) return fail(ctx, KZ_ERR_STATE, "the accel is not laid out level by level: call kzgpu_accel_build");
    const std::vector<uint32_t> &L = ctx->levels;
    const int nl = (int)L.size() - 1;
    /* once per built accel and device: every internal child one level down, every triangle in the record array */
    for (Device &d : ctx->devs) {
        KZ_CUDA(ctx, cudaSetDevice(d.id));
        KZ_CUDA(ctx, d.refit_flags.ensure(2 * sizeof(uint32_t)));
        KZ_CUDA(ctx, cudaMemsetAsync(d.refit_flags.p, 0, 2 * sizeof(uint32_t), d.stream));
        if (d.levels_checked || d.sc.n_nodes == 0) continue;
        for (int l = 0; l < nl; ++l) {
            const uint32_t next_hi = l + 1 < nl ? L[(size_t)l + 2] : L[(size_t)l + 1];
            k_refit_check<<<grid_for(L[(size_t)l + 1] - L[(size_t)l], 256, d.sm_count), 256, 0, d.stream>>>(d.sc.nodes, L[(size_t)l], L[(size_t)l + 1], L[(size_t)l + 1], next_hi,
                                                                                                          d.sc.n_tris, d.refit_flags.as<uint32_t>() + 1);
            ++d.launches;
        }
        KZ_CUDA(ctx, cudaGetLastError());
    }
    for (Device &d : ctx->devs) {
        if (d.levels_checked || d.sc.n_nodes == 0) continue;
        uint32_t bad = 0;
        KZ_CUDA(ctx, cudaSetDevice(d.id));
        KZ_CUDA(ctx, cudaMemcpyAsync(&bad, d.refit_flags.as<uint32_t>() + 1, 4, cudaMemcpyDeviceToHost, d.stream));
        KZ_CUDA(ctx, cudaStreamSynchronize(d.stream));
        if (bad || L.back() != d.sc.n_nodes) return fail(ctx, KZ_ERR_STATE, "the accel is not laid out level by level: call kzgpu_accel_build");
        d.levels_checked = true;
    }
    /* every device refits its own copy (the same records and vertices everywhere, exact arithmetic: the same bytes) */
    for (Device &d : ctx->devs) {
        if (d.sc.n_nodes == 0) continue;
        KZ_CUDA(ctx, cudaSetDevice(d.id));
        KZ_CUDA(ctx, d.refit_boxes.ensure((size_t)d.sc.n_nodes * sizeof(KzBox)));
        KzF4 *tris = d.accel.tris.as<KzF4>();
        KzNode8 *nodes = d.accel.nodes.as<KzNode8>();
        k_refit_tris<<<grid_for(d.sc.n_tris, 256, d.sm_count), 256, 0, d.stream>>>(d.sc.meshes, d.sc.vertices, d.sc.indices, tris, d.sc.n_tris, d.refit_flags.as<uint32_t>());
        for (int l = nl - 1; l >= 0; --l)
            k_refit_level<<<grid_for(L[(size_t)l + 1] - L[(size_t)l], 128, d.sm_count), 128, 0, d.stream>>>(nodes, tris, d.refit_boxes.as<KzBox>(), L[(size_t)l], L[(size_t)l + 1]);
        d.launches += 1 + (uint64_t)nl;
        KZ_CUDA(ctx, cudaGetLastError());
    }
    for (Device &d : ctx->devs) {
        if (d.sc.n_nodes == 0) continue;
        uint32_t mabs = 0;
        KZ_CUDA(ctx, cudaSetDevice(d.id));
        KZ_CUDA(ctx, cudaMemcpyAsync(&mabs, d.refit_flags.p, 4, cudaMemcpyDeviceToHost, d.stream));
        KZ_CUDA(ctx, cudaStreamSynchronize(d.stream));
        d.sc.scene_max_abs = d.accel.max_abs = kzlbvh::ord2f(mabs);
    }
    KZ_CUDA(ctx, cudaSetDevice(ctx->devs[0].id));
    ctx->built = true;
    return KZ_OK;
}

int kzgpu_camera_update(kzgpu_ctx *ctx, const kz_camera_desc *camera) {
    if (!ctx) return fail(nullptr, KZ_ERR_INVALID, "null context");
    if (!ctx->uploaded) return fail(ctx, KZ_ERR_STATE, "no scene uploaded");
    if (!camera) return fail(ctx, KZ_ERR_INVALID, "null camera");
    if (camera->width <= 0 || camera->height <= 0 || camera->width > 65535 || camera->height > 65535) return fail(ctx, KZ_ERR_INVALID, "camera size out of range");
    if (camera->width != ctx->hs->sc.camera.width || camera->height != ctx->hs->sc.camera.height)
        return fail(ctx, KZ_ERR_INVALID, "camera size differs from the uploaded one (the frame and the primary-hit hints are sized by it)");
    ctx->hs->sc.camera = *camera;
    for (Device &d : ctx->devs) d.sc.camera = *camera;
    return KZ_OK;
}

int kzgpu_accel_dump(kzgpu_ctx *ctx, int device, void *nodes, void *tris) {
    if (!ctx) return fail(nullptr, KZ_ERR_INVALID, "null context");
    if (!ctx->uploaded) return fail(ctx, KZ_ERR_STATE, "no scene uploaded");
    Device *d;
    int rc;
    if ((rc = select(ctx, device, &d))) return rc;
    if (!d->has_accel) return fail(ctx, KZ_ERR_STATE, "no accel built since the last upload");
    if ((d->sc.n_nodes && !nodes) || (d->sc.n_tris && !tris)) return fail(ctx, KZ_ERR_INVALID, "null buffer");
    if (d->sc.n_nodes) KZ_CUDA(ctx, cudaMemcpyAsync(nodes, d->sc.nodes, (size_t)d->sc.n_nodes * sizeof(KzNode8), cudaMemcpyDeviceToHost, d->stream));
    if (d->sc.n_tris) KZ_CUDA(ctx, cudaMemcpyAsync(tris, d->sc.tris, (size_t)d->sc.n_tris * 3 * sizeof(KzF4), cudaMemcpyDeviceToHost, d->stream));
    KZ_CUDA(ctx, cudaStreamSynchronize(d->stream));
    return KZ_OK;
}

int kzgpu_trace_device(kzgpu_ctx *ctx, int device, const void *d_rays, size_t n, int shadow, void *d_hits, void *stream) {
    (void)shadow;   /* accel.cpp:98-104: the shadow variant is the same closest-hit query */
    int rc = check_ready(ctx, true);
    if (rc) return rc;
    Device *d;
    if ((rc = select(ctx, device, &d))) return rc;
    if (n == 0) return KZ_OK;
    if (n > 0x7FFFFFFFull) return fail(ctx, KZ_ERR_INVALID, "batch larger than 2^31-1 rays");
    if (!d_rays || !d_hits) return fail(ctx, KZ_ERR_INVALID, "null ray/hit buffer");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    if (d->pending.size() > 8192) fold_events(*d);      /* callers that never poll kzgpu_stats: bound the live timing events */
    KZ_CUDA(ctx, cudaMemsetAsync(d->cursor.p, 0, 4, s));
    {
        Timed t(*d, s, CAT_TRACE);
        k_trace<<<d->grid_trace, KZ_TRACE_THREADS, 0, s>>>(d->sc, reinterpret_cast<const KzF4 *>(d_rays), (uint32_t)n, reinterpret_cast<float *>(d_hits), d->cursor.as<uint32_t>(), d->ctl);
        ++d->launches;
    }
    KZ_CUDA(ctx, cudaGetLastError());
    return KZ_OK;
}

int kzgpu_trace(kzgpu_ctx *ctx, int device, const kz_ray *rays, size_t n, int shadow, kz_hit *hits) {
    int rc = check_ready(ctx, true);
    if (rc) return rc;
    Device *d;
    if ((rc = select(ctx, device, &d))) return rc;
    if (n == 0) return KZ_OK;
    if (!rays || !hits) return fail(ctx, KZ_ERR_INVALID, "null ray/hit buffer");
    if (n > 0x7FFFFFFFull) return fail(ctx, KZ_ERR_INVALID, "batch larger than 2^31-1 rays");
    KZ_CUDA(ctx, d->scratch[0].ensure(n * sizeof(kz_ray), SCRATCH_MIN));
    KZ_CUDA(ctx, d->scratch[1].ensure(n * sizeof(kz_hit), SCRATCH_MIN));
    /* Three-stage pipeline over ray chunks: H2D of chunk c+1, traversal of chunk c and D2H of chunk c-1 run
     * concurrently (PCIe is full duplex; with pinned host buffers the call costs max(copy, trace), not the sum). */
    if (!d->copy_in) KZ_CUDA(ctx, cudaStreamCreateWithFlags(&d->copy_in.h, cudaStreamNonBlocking));
    if (!d->copy_out) KZ_CUDA(ctx, cudaStreamCreateWithFlags(&d->copy_out.h, cudaStreamNonBlocking));
    static const size_t n_chunks = [] { const char *e = getenv("KZGPU_TRACE_CHUNKS"); const int k = e ? atoi(e) : 16; return (size_t)(k < 1 ? 1 : (k > 256 ? 256 : k)); }();
    const size_t chunk = std::min<size_t>(n, std::max<size_t>(1u << 20, (n + n_chunks - 1) / n_chunks));
    /* The call ends with the traversal and the D2H copy of the LAST chunk, which nothing overlaps (and starts with the H2D copy of the
     * first): the chunks at both ends are therefore 1/8, 1/4 and 1/2 of the steady size (smaller ones lose more to the ~18 us ramp and
     * tail of a persistent launch than they win). */
    std::vector<size_t> sizes;
    {
        const size_t ramp[3] = {chunk / 8, chunk / 4, chunk / 2};
        const size_t ends = 2 * (ramp[0] + ramp[1] + ramp[2]);
        const char *ge = getenv("KZGPU_TRACE_GRADED");
        const bool graded = !ge || atoi(ge) != 0;
        if (graded && ramp[0] >= (1u << 16) && n >= ends + chunk) {
            for (int k = 0; k < 3; ++k) sizes.push_back(ramp[k]);
            size_t mid = n - ends;
            const size_t parts = (mid + chunk - 1) / chunk;
            for (size_t k = 0; k < parts; ++k) { const size_t c = (mid + (parts - k) - 1) / (parts - k); sizes.push_back(c); mid -= c; }
            for (int k = 2; k >= 0; --k) sizes.push_back(ramp[k]);
        } else {
            for (size_t first = 0; first < n; first += chunk) sizes.push_back(std::min(chunk, n - first));
        }
    }
    std::vector<cudaEvent_t> evs;
    char *d_rays = reinterpret_cast<char *>(d->scratch[0].p), *d_hits = reinterpret_cast<char *>(d->scratch[1].p);
    size_t first = 0;
    for (size_t ci = 0; ci < sizes.size() && rc == KZ_OK; first += sizes[ci], ++ci) {
        const size_t cnt = sizes[ci];
        cudaEvent_t e_in = get_event(*d), e_k = get_event(*d);
        evs.push_back(e_in); evs.push_back(e_k);
        cudaMemcpyAsync(d_rays + first * sizeof(kz_ray), rays + first, cnt * sizeof(kz_ray), cudaMemcpyHostToDevice, d->copy_in);
        cudaEventRecord(e_in, d->copy_in);
        cudaStreamWaitEvent(d->stream, e_in, 0);
        rc = kzgpu_trace_device(ctx, device, d_rays + first * sizeof(kz_ray), cnt, shadow, d_hits + first * sizeof(kz_hit), d->stream);
        cudaEventRecord(e_k, d->stream);
        cudaStreamWaitEvent(d->copy_out, e_k, 0);
        cudaMemcpyAsync(hits + first, d_hits + first * sizeof(kz_hit), cnt * sizeof(kz_hit), cudaMemcpyDeviceToHost, d->copy_out);
    }
    const cudaError_t e1 = cudaStreamSynchronize(d->copy_out), e2 = cudaStreamSynchronize(d->stream), e3 = cudaStreamSynchronize(d->copy_in);
    for (cudaEvent_t e : evs) d->free_events.push_back(e);
    if (rc) return rc;
    KZ_CUDA(ctx, e1); KZ_CUDA(ctx, e2); KZ_CUDA(ctx, e3);
    return KZ_OK;
}

int kzgpu_occluded(kzgpu_ctx *ctx, int device, const kz_ray *rays, size_t n, float trace_bias, uint8_t *occluded, uint8_t *segments) {
    int rc = check_ready(ctx, true);
    if (rc) return rc;
    Device *d;
    if ((rc = select(ctx, device, &d))) return rc;
    if (n == 0) return KZ_OK;
    if (n > 0x7FFFFFFFull) return fail(ctx, KZ_ERR_INVALID, "batch larger than 2^31-1 rays");
    if (!rays || !occluded) return fail(ctx, KZ_ERR_INVALID, "null buffer");
    KZ_CUDA(ctx, d->scratch[0].ensure(n * sizeof(kz_ray), SCRATCH_MIN));
    KZ_CUDA(ctx, d->scratch[1].ensure(2 * n, SCRATCH_MIN));
    uint8_t *d_occ = reinterpret_cast<uint8_t *>(d->scratch[1].p);
    KZ_CUDA(ctx, cudaMemcpyAsync(d->scratch[0].p, rays, n * sizeof(kz_ray), cudaMemcpyHostToDevice, d->stream));
    if (d->pending.size() > 8192) fold_events(*d);
    KZ_CUDA(ctx, cudaMemsetAsync(d->cursor.p, 0, 4, d->stream));
    {
        Timed t(*d, d->stream, CAT_TRACE);
        k_occluded<<<d->grid_occ, KZ_TRACE_THREADS, 0, d->stream>>>(d->sc, reinterpret_cast<const KzF4 *>(d->scratch[0].p), (uint32_t)n, trace_bias, d_occ, d_occ + n,
                                                                    d->cursor.as<uint32_t>(), d->ctl);
        ++d->launches;
    }
    KZ_CUDA(ctx, cudaMemcpyAsync(occluded, d_occ, n, cudaMemcpyDeviceToHost, d->stream));
    if (segments) KZ_CUDA(ctx, cudaMemcpyAsync(segments, d_occ + n, n, cudaMemcpyDeviceToHost, d->stream));
    KZ_CUDA(ctx, cudaStreamSynchronize(d->stream));
    return KZ_OK;
}

int kzgpu_sample_dump(kzgpu_ctx *ctx, const int32_t *triples, size_t n, const char *pattern, float *out) {
    int rc = check_ready(ctx, false);
    if (rc) return rc;
    Device *d;
    if ((rc = select(ctx, 0, &d))) return rc;
    if (!pattern || (!triples && n) || (!out && n)) return fail(ctx, KZ_ERR_INVALID, "null argument");
    size_t per = 0, plen = strlen(pattern);
    for (const char *p = pattern; *p; ++p) {
        if (*p != '1' && *p != '2' && *p != 'P') return fail(ctx, KZ_ERR_INVALID, "pattern may only contain '1', '2', 'P'");
        per += (*p == '1') ? 1 : 2;
    }
    if (n == 0 || per == 0) return KZ_OK;
    KZ_CUDA(ctx, d->scratch[0].ensure(n * 12, SCRATCH_MIN));
    KZ_CUDA(ctx, d->scratch[1].ensure(n * per * 4, SCRATCH_MIN));
    KZ_CUDA(ctx, d->scratch[2].ensure(plen + 1, SCRATCH_MIN));
    KZ_CUDA(ctx, cudaMemcpyAsync(d->scratch[0].p, triples, n * 12, cudaMemcpyHostToDevice, d->stream));
    KZ_CUDA(ctx, cudaMemcpyAsync(d->scratch[2].p, pattern, plen + 1, cudaMemcpyHostToDevice, d->stream));
    k_sample_dump<<<(unsigned)((n + 127) / 128), 128, 0, d->stream>>>(d->sc, reinterpret_cast<const int32_t *>(d->scratch[0].p), (uint32_t)n,
                                                                      reinterpret_cast<const char *>(d->scratch[2].p), (uint32_t)per, reinterpret_cast<float *>(d->scratch[1].p));
    ++d->launches;
    KZ_CUDA(ctx, cudaMemcpyAsync(out, d->scratch[1].p, n * per * 4, cudaMemcpyDeviceToHost, d->stream));
    KZ_CUDA(ctx, cudaStreamSynchronize(d->stream));
    return KZ_OK;
}

int kzgpu_camera_rays(kzgpu_ctx *ctx, const float *samples4, size_t n, kz_ray *out) {
    int rc = check_ready(ctx, false);
    if (rc) return rc;
    Device *d;
    if ((rc = select(ctx, 0, &d))) return rc;
    if (n == 0) return KZ_OK;
    if (!samples4 || !out) return fail(ctx, KZ_ERR_INVALID, "null argument");
    KZ_CUDA(ctx, d->scratch[0].ensure(n * 16, SCRATCH_MIN));
    KZ_CUDA(ctx, d->scratch[1].ensure(n * 32, SCRATCH_MIN));
    KZ_CUDA(ctx, cudaMemcpyAsync(d->scratch[0].p, samples4, n * 16, cudaMemcpyHostToDevice, d->stream));
    k_camera_rays<<<(unsigned)((n + 127) / 128), 128, 0, d->stream>>>(d->sc, reinterpret_cast<const KzF4 *>(d->scratch[0].p), (uint32_t)n, reinterpret_cast<KzF4 *>(d->scratch[1].p));
    ++d->launches;
    KZ_CUDA(ctx, cudaMemcpyAsync(out, d->scratch[1].p, n * 32, cudaMemcpyDeviceToHost, d->stream));
    KZ_CUDA(ctx, cudaStreamSynchronize(d->stream));
    return KZ_OK;
}

int kzgpu_bsdf_query(kzgpu_ctx *ctx, int bsdf, int mode, const float wi[3], const float wo[3], const float uv[2], float accumulated_roughness,
                     float sample1, const float sample2[2], float out[8]) {
    int rc = check_ready(ctx, false);
    if (rc) return rc;
    Device *d;
    if ((rc = select(ctx, 0, &d))) return rc;
    KzBsdfQuery q;
    memset(&q, 0, sizeof(q));
    q.mesh = -1;
    for (size_t g = 0; g < ctx->hs->meshes.size(); ++g) if (ctx->hs->meshes[g].bsdf == bsdf) { q.mesh = (int32_t)g; break; }
    if (q.mesh < 0) return fail(ctx, KZ_ERR_INVALID, "no mesh uses this bsdf");
    for (int k = 0; k < 3; ++k) { q.wi[k] = wi[k]; q.wo[k] = wo ? wo[k] : 0.f; }
    q.uv[0] = uv[0]; q.uv[1] = uv[1]; q.acc_rough = accumulated_roughness; q.s1 = sample1;
    q.s2[0] = sample2 ? sample2[0] : 0.f; q.s2[1] = sample2 ? sample2[1] : 0.f; q.mode = mode;
    KZ_CUDA(ctx, d->scratch[0].ensure(sizeof(q), SCRATCH_MIN));
    KZ_CUDA(ctx, d->scratch[1].ensure(32, SCRATCH_MIN));
    KZ_CUDA(ctx, cudaMemcpyAsync(d->scratch[0].p, &q, sizeof(q), cudaMemcpyHostToDevice, d->stream));
    k_bsdf_query<<<1, 32, 0, d->stream>>>(d->sc, reinterpret_cast<const KzBsdfQuery *>(d->scratch[0].p), 1u, reinterpret_cast<float *>(d->scratch[1].p));
    ++d->launches;
    KZ_CUDA(ctx, cudaMemcpyAsync(out, d->scratch[1].p, 32, cudaMemcpyDeviceToHost, d->stream));
    KZ_CUDA(ctx, cudaStreamSynchronize(d->stream));
    return KZ_OK;
}

int kzgpu_image_lookup(kzgpu_ctx *ctx, int image, int level, const float *st, size_t n, float *rgb) {
    int rc = check_ready(ctx, false);
    if (rc) return rc;
    Device *d;
    if ((rc = select(ctx, 0, &d))) return rc;
    if (image < 0 || image >= (int)ctx->hs->images.size()) return fail(ctx, KZ_ERR_INVALID, "image index out of range");
    if (level < 0) return fail(ctx, KZ_ERR_INVALID, "negative mip level");
    if (n == 0) return KZ_OK;
    if (!st || !rgb) return fail(ctx, KZ_ERR_INVALID, "null argument");
    KZ_CUDA(ctx, d->scratch[0].ensure(n * 8, SCRATCH_MIN));
    KZ_CUDA(ctx, d->scratch[1].ensure(n * 12, SCRATCH_MIN));
    KzScene sc = d->sc;
    int lookup_image = image;
    DevMem pyr_mem, rec_mem;
    if (level > 0) {
        /* the renderer only reads level 0 (ImageTexture::eval passes zero derivatives, texture.cpp:52-57), so the pyramid is not
         * kept resident: it is built here, for this image, by 2x2 box filtering on the device */
        const KzImageRec im = ctx->hs->images[(size_t)image];
        KzImageRec pr = im; pr.texel_offset = 0; pr.n_levels = 0;
        size_t total = (size_t)im.width * im.height;
        for (int w = im.width, h = im.height; w > 1 || h > 1;) { w = w > 1 ? w >> 1 : 1; h = h > 1 ? h >> 1 : 1; total += (size_t)w * h; ++pr.n_levels; }
        KzF4 *pyr = nullptr; KzImageRec *rec = nullptr;
        if ((rc = dev_alloc(ctx, pyr_mem, total, &pyr)) || (rc = dev_alloc(ctx, rec_mem, 1, &rec))) return rc;
        cudaError_t e = cudaMemcpyAsync(pyr, d->sc.texels + im.texel_offset, (size_t)im.width * im.height * sizeof(KzF4), cudaMemcpyDeviceToDevice, d->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(rec, &pr, sizeof(pr), cudaMemcpyHostToDevice, d->stream);
        KZ_CUDA(ctx, e);
        size_t src = 0; int sw = im.width, sh = im.height;
        for (int l = 1; l <= pr.n_levels; ++l) {
            const int dw = sw > 1 ? sw >> 1 : 1, dh = sh > 1 ? sh >> 1 : 1;
            const size_t dst = src + (size_t)sw * sh;
            dim3 blk(32, 8), grd((unsigned)(dw + 31) / 32, (unsigned)(dh + 7) / 8);
            k_mip_level<<<grd, blk, 0, d->stream>>>(pyr, src, sw, sh, dst, dw, dh);
            ++d->launches;
            src = dst; sw = dw; sh = dh;
        }
        sc.texels = pyr; sc.images = rec; lookup_image = 0;
    }
    cudaError_t e = cudaMemcpyAsync(d->scratch[0].p, st, n * 8, cudaMemcpyHostToDevice, d->stream);
    if (e == cudaSuccess) {
        k_image_lookup<<<(unsigned)((n + 127) / 128), 128, 0, d->stream>>>(sc, lookup_image, level, reinterpret_cast<const float *>(d->scratch[0].p), (uint32_t)n,
                                                                           reinterpret_cast<float *>(d->scratch[1].p));
        ++d->launches;
        e = cudaMemcpyAsync(rgb, d->scratch[1].p, n * 12, cudaMemcpyDeviceToHost, d->stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(d->stream);
    KZ_CUDA(ctx, e);
    return KZ_OK;
}

int kzgpu_intersection_dump(kzgpu_ctx *ctx, const kz_ray *rays, size_t n, float *out24) {
    int rc = check_ready(ctx, true);
    if (rc) return rc;
    Device *d;
    if ((rc = select(ctx, 0, &d))) return rc;
    if (n == 0) return KZ_OK;
    if (!rays || !out24) return fail(ctx, KZ_ERR_INVALID, "null argument");
    if (n > 0x7FFFFFFFull) return fail(ctx, KZ_ERR_INVALID, "batch larger than 2^31-1 rays");
    KZ_CUDA(ctx, d->scratch[0].ensure(n * sizeof(kz_ray), SCRATCH_MIN));
    KZ_CUDA(ctx, d->scratch[1].ensure(n * 96, SCRATCH_MIN));
    KZ_CUDA(ctx, cudaMemcpyAsync(d->scratch[0].p, rays, n * sizeof(kz_ray), cudaMemcpyHostToDevice, d->stream));
    k_intersection_dump<<<(unsigned)((n + KZ_TRACE_THREADS - 1) / KZ_TRACE_THREADS), KZ_TRACE_THREADS, 0, d->stream>>>(d->sc, reinterpret_cast<const KzF4 *>(d->scratch[0].p), (uint32_t)n,
                                                                                                                    reinterpret_cast<float *>(d->scratch[1].p));
    ++d->launches;
    KZ_CUDA(ctx, cudaMemcpyAsync(out24, d->scratch[1].p, n * 96, cudaMemcpyDeviceToHost, d->stream));
    KZ_CUDA(ctx, cudaStreamSynchronize(d->stream));
    return KZ_OK;
}

int kzgpu_light_sample_dump(kzgpu_ctx *ctx, const float *ref3, const float *u5, size_t n, float *out16) {
    int rc = check_ready(ctx, false);
    if (rc) return rc;
    Device *d;
    if ((rc = select(ctx, 0, &d))) return rc;
    if (n == 0) return KZ_OK;
    if (!ref3 || !u5 || !out16) return fail(ctx, KZ_ERR_INVALID, "null argument");
    if (n > 0x7FFFFFFFull) return fail(ctx, KZ_ERR_INVALID, "batch too large");
    KZ_CUDA(ctx, d->scratch[0].ensure(n * 12, SCRATCH_MIN));
    KZ_CUDA(ctx, d->scratch[1].ensure(n * 64, SCRATCH_MIN));
    KZ_CUDA(ctx, d->scratch[2].ensure(n * 20, SCRATCH_MIN));
    KZ_CUDA(ctx, cudaMemcpyAsync(d->scratch[0].p, ref3, n * 12, cudaMemcpyHostToDevice, d->stream));
    KZ_CUDA(ctx, cudaMemcpyAsync(d->scratch[2].p, u5, n * 20, cudaMemcpyHostToDevice, d->stream));
    k_light_sample_dump<<<(unsigned)((n + 127) / 128), 128, 0, d->stream>>>(d->sc, reinterpret_cast<const float *>(d->scratch[0].p), reinterpret_cast<const float *>(d->scratch[2].p),
                                                                            (uint32_t)n, reinterpret_cast<float *>(d->scratch[1].p));
    ++d->launches;
    KZ_CUDA(ctx, cudaMemcpyAsync(out16, d->scratch[1].p, n * 64, cudaMemcpyDeviceToHost, d->stream));
    KZ_CUDA(ctx, cudaStreamSynchronize(d->stream));
    return KZ_OK;
}

int kzgpu_frame_dims(const kzgpu_ctx *ctx, int32_t *width, int32_t *height, int32_t *border) {
    if (!ctx || !ctx->hs) return fail(nullptr, KZ_ERR_STATE, "no scene uploaded");
    if (width) *width = ctx->hs->sc.camera.width;
    if (height) *height = ctx->hs->sc.camera.height;
    if (border) *border = ctx->hs->sc.border;
    return KZ_OK;
}

static int check_req(kzgpu_ctx *ctx, const kz_render_req *req) {
    if (!req) return fail(ctx, KZ_ERR_INVALID, "null request");
    const kz_camera_desc &c = ctx->hs->sc.camera;
    if (req->x0 < 0 || req->y0 < 0 || req->x1 > c.width || req->y1 > c.height || req->x0 > req->x1 || req->y0 > req->y1)
        return fail(ctx, KZ_ERR_INVALID, "render rectangle outside the film");
    if (req->spp_begin < 0 || req->spp_end < req->spp_begin) return fail(ctx, KZ_ERR_INVALID, "bad sample range");
    /* pmj02bn reads per-pixel sample tables of sample_count entries (sampler.cpp:290-314,333-337): an index beyond is out of bounds */
    if (ctx->hs->sc.sampler_type == KZ_SAMPLER_PMJ02BN && (uint32_t)req->spp_end > ctx->hs->sc.sample_count)
        return fail(ctx, KZ_ERR_INVALID, "sample range exceeds the pmj02bn sampler's sample_count");
    return KZ_OK;
}

int kzgpu_render_device(kzgpu_ctx *ctx, int device, const kz_render_req *req, void **d_frame_inout, void *stream) {
    int rc = check_ready(ctx, true);
    if (rc) return rc;
    if ((rc = check_req(ctx, req))) return rc;
    Device *d;
    if ((rc = select(ctx, device, &d))) return rc;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    /* caller-owned frame (e.g. a torch tensor that an NCCL reduce follows) for this call, or the context's own */
    if (d_frame_inout && *d_frame_inout) d->frame = reinterpret_cast<KzF4 *>(*d_frame_inout);
    if (req->clear_frame) {
        cudaError_t e = cudaMemsetAsync(d->frame, 0, d->frame_texels * sizeof(KzF4), s);
        if (e != cudaSuccess) { d->frame = d->frame_mem.as<KzF4>(); return fail(ctx, KZ_ERR_CUDA, std::string("cudaMemsetAsync(frame): ") + cudaGetErrorString(e)); }
    }
    rc = enqueue_render(ctx, ctx, *d, *req, s);
    if (d_frame_inout) *d_frame_inout = d->frame;
    d->frame = d->frame_mem.as<KzF4>();
    return rc;
}

int kzgpu_render(kzgpu_ctx *ctx, const kz_render_req *req, float *frame_rgbw) {
    int rc = check_ready(ctx, true);
    if (rc) return rc;
    if ((rc = check_req(ctx, req))) return rc;
    if (!frame_rgbw) return fail(ctx, KZ_ERR_INVALID, "null frame");
    const int nd = (int)ctx->devs.size();
    const int nS = req->spp_end - req->spp_begin;
    const size_t texels = ctx->devs[0].frame_texels;
    /* shard by sample index (SURVEY 8e): device g takes a contiguous slice of [spp_begin, spp_end).  One host thread per
     * device: a long render is thousands of launches, and a single thread would block on the first device's launch queue
     * before it ever reaches the second one.  Workers report through their own slot (never through ctx->error). */
    std::vector<int> rcs((size_t)nd, KZ_OK);
    std::vector<std::string> errs((size_t)nd);
    auto work = [&](int g) {
        Device &d = ctx->devs[(size_t)g];
        auto bail = [&](cudaError_t e, const char *what) { rcs[(size_t)g] = KZ_ERR_CUDA; errs[(size_t)g] = std::string(what) + ": " + cudaGetErrorString(e); };
        cudaError_t e = cudaSetDevice(d.id);
        if (e != cudaSuccess) return bail(e, "cudaSetDevice");
        kz_render_req r = *req;
        r.spp_begin = req->spp_begin + (int)((long long)nS * g / nd);
        r.spp_end = req->spp_begin + (int)((long long)nS * (g + 1) / nd);
        /* the root's frame starts from the caller's frame when the request accumulates (progressive / resumed renders) */
        if (g == 0 && !req->clear_frame) e = cudaMemcpyAsync(d.frame, frame_rgbw, texels * sizeof(KzF4), cudaMemcpyHostToDevice, d.stream);
        else e = cudaMemsetAsync(d.frame, 0, texels * sizeof(KzF4), d.stream);
        if (e != cudaSuccess) return bail(e, "frame initialisation");
        const int rc = enqueue_render(ctx, nullptr, d, r, d.stream);
        if (rc != KZ_OK) { rcs[(size_t)g] = rc; errs[(size_t)g] = g_error; return; }
        if ((e = cudaEventRecord(d.splat_done, d.stream)) != cudaSuccess) return bail(e, "cudaEventRecord");
    };
    std::vector<std::thread> pool;
    for (int g = 1; g < nd; ++g) pool.emplace_back(work, g);
    work(0);
    for (std::thread &t : pool) t.join();
    for (int g = 0; g < nd; ++g)
        if (rcs[(size_t)g] != KZ_OK) {
            for (Device &d : ctx->devs) { cudaSetDevice(d.id); cudaStreamSynchronize(d.stream); }
            return fail(ctx, rcs[(size_t)g], "device " + std::to_string(g) + ": " + errs[(size_t)g]);
        }
    Device &root = ctx->devs[0];
    if (nd > 1) {
        /* ImageBlock::put(ImageBlock&) (block.cpp:87-96) over NVLink: once every device finished splatting, device g sums slice g of
         * all frames through peer loads and stores it into the root's frame; the root then holds the merged frame */
        KzFramePtrs fp;
        for (int g = 0; g < nd; ++g) fp.f[g] = ctx->devs[(size_t)g].frame;
        for (int g = 0; g < nd; ++g) {
            Device &d = ctx->devs[(size_t)g];
            KZ_CUDA(ctx, cudaSetDevice(d.id));
            for (int o = 0; o < nd; ++o) if (o != g) KZ_CUDA(ctx, cudaStreamWaitEvent(d.stream, ctx->devs[(size_t)o].splat_done, 0));
            const size_t begin = texels * (size_t)g / (size_t)nd, end = texels * (size_t)(g + 1) / (size_t)nd;
            if (end > begin) {
                Timed t(d, d.stream, CAT_MERGE);
                k_frame_reduce<<<grid_for(end - begin, 256, d.sm_count), 256, 0, d.stream>>>(fp, nd, begin, end);
                ++d.launches;
            }
            KZ_CUDA(ctx, cudaEventRecord(d.merge_done, d.stream));
        }
        KZ_CUDA(ctx, cudaSetDevice(root.id));
        for (int g = 1; g < nd; ++g) KZ_CUDA(ctx, cudaStreamWaitEvent(root.stream, ctx->devs[(size_t)g].merge_done, 0));
    }
    KZ_CUDA(ctx, cudaSetDevice(root.id));
    KZ_CUDA(ctx, cudaMemcpyAsync(frame_rgbw, root.frame, texels * sizeof(KzF4), cudaMemcpyDeviceToHost, root.stream));
    KZ_CUDA(ctx, cudaStreamSynchronize(root.stream));
    /* the peers may not start their next request (which clears their frame) before the root has read it */
    for (int g = 1; g < nd; ++g) { KZ_CUDA(ctx, cudaSetDevice(ctx->devs[(size_t)g].id)); KZ_CUDA(ctx, cudaStreamSynchronize(ctx->devs[(size_t)g].stream)); }
    KZ_CUDA(ctx, cudaSetDevice(root.id));
    return KZ_OK;
}

int kzgpu_resolve(kzgpu_ctx *ctx, const float *frame_rgbw, float *rgb_linear, uint8_t *srgb8) {
    int rc = check_ready(ctx, false);
    if (rc) return rc;
    Device *d;
    if ((rc = select(ctx, 0, &d))) return rc;
    if (!frame_rgbw) return fail(ctx, KZ_ERR_INVALID, "null frame");
    const KzScene &sc = d->sc;
    const int W = sc.camera.width, H = sc.camera.height;
    const size_t npx = (size_t)W * H;
    KZ_CUDA(ctx, d->scratch[0].ensure(d->frame_texels * sizeof(KzF4), SCRATCH_MIN));
    KZ_CUDA(ctx, d->scratch[1].ensure(npx * 12, SCRATCH_MIN));
    KZ_CUDA(ctx, d->scratch[2].ensure(npx * 3, SCRATCH_MIN));
    KZ_CUDA(ctx, cudaMemcpyAsync(d->scratch[0].p, frame_rgbw, d->frame_texels * sizeof(KzF4), cudaMemcpyHostToDevice, d->stream));
    dim3 blk(32, 8), grd((unsigned)(W + 31) / 32, (unsigned)(H + 7) / 8);
    k_resolve<<<grd, blk, 0, d->stream>>>(reinterpret_cast<const KzF4 *>(d->scratch[0].p), W, H, sc.border, rgb_linear ? reinterpret_cast<float *>(d->scratch[1].p) : nullptr,
                                          srgb8 ? reinterpret_cast<uint8_t *>(d->scratch[2].p) : nullptr);
    ++d->launches;
    if (rgb_linear) KZ_CUDA(ctx, cudaMemcpyAsync(rgb_linear, d->scratch[1].p, npx * 12, cudaMemcpyDeviceToHost, d->stream));
    if (srgb8) KZ_CUDA(ctx, cudaMemcpyAsync(srgb8, d->scratch[2].p, npx * 3, cudaMemcpyDeviceToHost, d->stream));
    KZ_CUDA(ctx, cudaStreamSynchronize(d->stream));
    return KZ_OK;
}

int kzgpu_configure(kzgpu_ctx *ctx, const char *key, int value) {
    if (!ctx || !key) return fail(ctx, KZ_ERR_INVALID, "null argument");
    const std::string k(key);
    if (k == "lanes") { if (value < 1 || value > KZ_MAX_LANES) return fail(ctx, KZ_ERR_INVALID, "lanes must be 1.." + std::to_string(KZ_MAX_LANES)); ctx->lanes = value; return KZ_OK; }
    if (k == "pool_log2") { if (value < 10 || value > 26) return fail(ctx, KZ_ERR_INVALID, "pool_log2 must be 10..26"); ctx->pool_cap = 1u << value; return KZ_OK; }
    if (k == "spp_group") { if (value < 1) return fail(ctx, KZ_ERR_INVALID, "spp_group must be >= 1"); ctx->spp_group = value; return KZ_OK; }
    if (k == "primary_hint") { if (value < 0 || value > 2) return fail(ctx, KZ_ERR_INVALID, "primary_hint must be 0, 1 or 2"); ctx->primary_hint = value; return KZ_OK; }
    return fail(ctx, KZ_ERR_INVALID, "unknown option \"" + k + "\"");
}

int kzgpu_stats(kzgpu_ctx *ctx, kz_stats *out) {
    if (!ctx || !out) return fail(ctx, KZ_ERR_INVALID, "null argument");
    memset(out, 0, sizeof(*out));
    for (Device &d : ctx->devs) {
        KZ_CUDA(ctx, cudaSetDevice(d.id));
        KZ_CUDA(ctx, cudaDeviceSynchronize());
        fold_events(d);
        for (Lane &L : d.lane) {
            KzControl c;
            KZ_CUDA(ctx, cudaMemcpy(&c, L.ctl, sizeof(c), cudaMemcpyDeviceToHost));
            out->paths += c.paths; out->rays_extension += c.rays_ext; out->rays_shadow += c.rays_shadow; out->vertices += c.vertices;
            out->rays_seeded += c.rays_seeded;
        }
        out->kernel_launches += d.launches;
        out->ms_trace = std::max(out->ms_trace, d.ms[CAT_TRACE]);
        out->ms_shade = std::max(out->ms_shade, d.ms[CAT_SHADE]);
        out->ms_total = std::max(out->ms_total, d.ms[CAT_TOTAL]);
        out->ms_merge = std::max(out->ms_merge, d.ms[CAT_MERGE]);
    }
    out->bvh_nodes = ctx->bvh_nodes; out->bvh_bytes = ctx->bvh_bytes; out->ms_build = ctx->ms_build; out->ms_upload = ctx->ms_upload;
    return KZ_OK;
}

int kzgpu_stats_reset(kzgpu_ctx *ctx) {
    if (!ctx) return fail(nullptr, KZ_ERR_INVALID, "null context");
    for (Device &d : ctx->devs) {
        KZ_CUDA(ctx, cudaSetDevice(d.id));
        KZ_CUDA(ctx, cudaDeviceSynchronize());
        fold_events(d);
        for (double &m : d.ms) m = 0; d.launches = 0;
        /* keep queue state, zero the counters */
        for (Lane &L : d.lane) KZ_CUDA(ctx, cudaMemset(reinterpret_cast<char *>(L.ctl) + offsetof(KzControl, paths), 0, 5 * sizeof(unsigned long long)));
    }
    return KZ_OK;
}

}  // extern "C"
