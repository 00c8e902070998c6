/* kz_kernels.cuh -- the sm_100a kernels of the wavefront path tracer.
 *
 * Pipeline per chunk of path slots (kz_api.cu drives it without any host round trip):
 *
 *   k_chunk_reset -> k_raygen -> for bounce b = 0..maxDepth:
 *        k_bounce_reset -> k_extend (closest hit, sorts slots into material-class queues)
 *                       -> k_shade<TERMINAL|DIFFUSE|KISS|NORMALMAP> (one launch per class present)
 *                       -> k_shadow (closest-hit walk through invisible lights, adds the NEE term)
 *   -> k_accumulate (filtered splat into the bordered frame)
 *
 * Queues are arrays of slot indices with device-resident counters; every kernel is launched with
 * a persistent grid (SM count x resident CTAs) and reads its item count from HBM, so the host
 * never waits on a count.  Traversal kernels fetch 32-ray packets per warp through an atomic
 * cursor (rays differ wildly in cost); shading kernels use a static warp-strided assignment.
 * Pushes are warp-aggregated: one ballot + one atomicAdd per warp per queue.
 *
 * No tensor-core, TMA or cluster machinery on purpose: every stage is a data-dependent gather
 * (BVH nodes, triangles, vertex attributes) or per-item ALU work; there is no tile to stage.
 */
#ifndef KZ_KERNELS_CUH
#define KZ_KERNELS_CUH
#include "kz_path.h"

#ifndef KZ_TRACE_THREADS
#define KZ_TRACE_THREADS 128
#endif
#ifndef KZ_TRACE_MIN_BLOCKS
#define KZ_TRACE_MIN_BLOCKS 8       /* k_extend / k_shadow: 64 registers (a few spilled words); with two lanes in flight 8 CTAs/SM beat ptxas' 72-80 registers: 1074 -> 1093 Mpaths/s */
#endif
#ifndef KZ_BATCH_MIN_BLOCKS
#define KZ_BATCH_MIN_BLOCKS 8       /* k_trace / k_occluded: 8 CTAs of 128 threads = 64 registers, no spills (measured best) */
#endif
#define KZ_SHADE_THREADS 128

struct KzControl {
    /* [k]: low word = entries of the extension queue k (ping-pong), high word = entries of the shadow queue
     * filled by the same shade pass -- packed so one 64-bit atomic reserves space in both queues */
    unsigned long long ext_shadow[2];
    uint32_t n_class[KZ_NUM_CLASSES];     /* material-class queue counts                    */
    uint32_t head_ext, head_shadow, head_trace;   /* persistent-fetch cursors               */
    uint32_t pad[1];
    unsigned long long paths, rays_ext, rays_shadow, vertices, rays_seeded;
};

struct KzQueues {
    uint32_t *ext[2];
    uint32_t *cls[KZ_NUM_CLASSES];
    uint32_t *shadow;
};

struct KzChunk {
    int32_t x0, y0, x1, y1;          /* pixel rectangle                                     */
    uint32_t tiles_x;                /* 8x4 pixel tiles per row                             */
    uint32_t npx_padded;             /* tiles_x * tiles_y * 32                              */
    int32_t spp_begin;
    uint32_t n_spp;                  /* sample indices of the request                       */
    uint32_t spp_group;              /* consecutive sample indices of one tile that are neighbours in path order (1 = sample-major) */
    unsigned long long first;        /* first global path index of this chunk               */
    uint32_t count;                  /* slots used by this chunk                            */
};

#define KZ_FULL 0xFFFFFFFFu

__device__ __forceinline__ uint32_t kz_lane() { return threadIdx.x & 31u; }

/* Warp-aggregated append; must be reached by all 32 lanes of the warp. */
__device__ __forceinline__ void kz_push(uint32_t *queue, uint32_t *counter, bool pred, uint32_t value) {
    const uint32_t mask = __ballot_sync(KZ_FULL, pred);
    if (mask == 0u) return;
    const uint32_t lane = kz_lane();
    const uint32_t leader = (uint32_t)__ffs((int)mask) - 1u;
    uint32_t base = 0u;
    if (lane == leader) base = atomicAdd(counter, (uint32_t)__popc(mask));
    base = __shfl_sync(KZ_FULL, base, (int)leader);
    if (pred) queue[base + (uint32_t)__popc(mask & ((1u << lane) - 1u))] = value;
}

__device__ __forceinline__ uint32_t *kz_ext_counter(KzControl *ctl, int k) { return reinterpret_cast<uint32_t *>(&ctl->ext_shadow[k]); }
__device__ __forceinline__ uint32_t kz_ext_count(const KzControl *ctl, int k) { return (uint32_t)(ctl->ext_shadow[k] & 0xFFFFFFFFull); }
__device__ __forceinline__ uint32_t kz_shadow_count(const KzControl *ctl, int k) { return (uint32_t)(ctl->ext_shadow[k] >> 32); }

/* Appends `value` to queue A and/or queue B with ONE atomic per warp (counters packed lo|hi); all 32 lanes must call. */
__device__ __forceinline__ void kz_push2(uint32_t *qa, uint32_t *qb, unsigned long long *counter, bool pa, bool pb, uint32_t value) {
    const uint32_t ma = __ballot_sync(KZ_FULL, pa), mb = __ballot_sync(KZ_FULL, pb);
    if ((ma | mb) == 0u) return;
    const uint32_t lane = kz_lane(), lt = (1u << lane) - 1u;
    unsigned long long base = 0ull;
    if (lane == 0u) base = atomicAdd(counter, (unsigned long long)__popc(ma) | ((unsigned long long)__popc(mb) << 32));
    base = __shfl_sync(KZ_FULL, base, 0);
    if (pa) qa[(uint32_t)(base & 0xFFFFFFFFull) + (uint32_t)__popc(ma & lt)] = value;
    if (pb) qb[(uint32_t)(base >> 32) + (uint32_t)__popc(mb & lt)] = value;
}

/* Next 32-item packet of a queue for this warp (persistent threads). */
__device__ __forceinline__ uint32_t kz_fetch32(uint32_t *cursor) {
    uint32_t base = 0u;
    if (kz_lane() == 0u) base = atomicAdd(cursor, 32u);
    return __shfl_sync(KZ_FULL, base, 0);
}

__device__ __forceinline__ void kz_flush_counters(KzControl *ctl, const KzCounters &c) {
    unsigned long long e = c.rays_ext, s = c.rays_shadow, v = c.vertices, h = c.rays_seeded;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        e += __shfl_down_sync(KZ_FULL, e, o);
        s += __shfl_down_sync(KZ_FULL, s, o);
        v += __shfl_down_sync(KZ_FULL, v, o);
        h += __shfl_down_sync(KZ_FULL, h, o);
    }
    if (kz_lane() == 0u) {
        if (e) atomicAdd(&ctl->rays_ext, e);
        if (s) atomicAdd(&ctl->rays_shadow, s);
        if (v) atomicAdd(&ctl->vertices, v);
        if (h) atomicAdd(&ctl->rays_seeded, h);
    }
}

/* ---- warp-cooperative persistent traversal ----------------------------------------------------
 * One warp owns 32 ray slots.  Lanes whose ray is finished are refilled from the work queue (one
 * ballot + one atomicAdd per refill) once enough loop iterations have been lost to idle lanes
 * (Aila/Laine persistent threads; thresholds re-measured on B200: refill as soon as 8 lane-iterations are lost), and a lane postpones its
 * leaf tests (pushes the triangle group back on its stack) while fewer than 1/5 of the active lanes
 * have triangles to test, so node steps and Pluecker tests run with fuller warps.
 * Traversal order therefore differs per launch, results do not: ties resolve by (geomID, primID).
 *
 * Job: per-lane policy object.
 *   void begin(uint32_t item, KzRayIn &r)                   load the ray of work item `item`
 *   void seed(const KzScene &sc, KzTrav &t)                 called right after the traversal of that ray was initialised: may preset
 *                                                           its best hit (kz_trav_preset); not called for follow-up rays
 *   bool end(uint32_t item, const KzHit &h, KzRayIn &r)     consume the closest hit; return true and fill `r`
 *                                                           to continue the same item with a follow-up ray
 *   static constexpr bool kStopsEarly                       the job only asks WHETHER something opaque is hit (shadow rays)
 *   bool stop(const KzScene &sc, const KzTrav &t)           called after a triangle became the best hit: true ends the ray there */
struct KzRayIn { float ox, oy, oz, tmin, dx, dy, dz, tmax; };
#ifndef KZ_FETCH_ND
#define KZ_FETCH_ND 0
#endif
#ifndef KZ_FETCH_NW
#define KZ_FETCH_NW 8
#endif
#ifndef KZ_TRAV_MODE
#define KZ_TRAV_MODE 0          /* 0: one node step + postponed leaf tests per iteration; 1: while-while */
#endif
#ifndef KZ_WAIT_IDLE
#define KZ_WAIT_IDLE 1
#endif
#ifndef KZ_POSTPONE_NUM
#define KZ_POSTPONE_NUM 1       /* postpone leaf tests while active lanes < NUM/DEN of the lanes in the loop */
#define KZ_POSTPONE_DEN 5
#endif

template <class Job>
__device__ __forceinline__ void kz_warp_trace(const KzScene &sc, const KzStackRef &stk, uint32_t *cursor, uint32_t n, Job &job) {
    KzTrav t;
    KzLocalStack ls;
    t.sp = 0; t.ng_y = 0u; t.tg_y = 0u;
    bool active = false, finished = false, exhausted = false;
    uint32_t item = 0u;
    const uint32_t lane = kz_lane(), lt = (1u << lane) - 1u;
    for (;;) {
        /* The warp is converged here.  Lanes whose ray ended since the last visit consume their hit TOGETHER (job.end is the
         * expensive, divergent part of the extension and shadow jobs: post-intersection, state stores, queue pushes); doing it
         * at the moment a lane finishes ran it with one or two lanes active. */
        if (finished) {
            KzRayIn r;
            if (job.end(item, t.best, r)) kz_trav_init(sc, t, r.ox, r.oy, r.oz, r.dx, r.dy, r.dz, r.tmin, r.tmax);
            else active = false;
            finished = false;
        }
        if (!exhausted) {
            const uint32_t idle = __ballot_sync(KZ_FULL, !active);
            if (idle) {
                const uint32_t leader = (uint32_t)__ffs((int)idle) - 1u;
                uint32_t base = 0u;
                if (lane == leader) base = atomicAdd(cursor, (uint32_t)__popc(idle));
                base = __shfl_sync(KZ_FULL, base, (int)leader);
                if (!active) {
                    const uint32_t idx = base + (uint32_t)__popc(idle & lt);
                    if (idx < n) {
                        item = idx;
                        KzRayIn r;
                        job.begin(item, r);
                        kz_trav_init(sc, t, r.ox, r.oy, r.oz, r.dx, r.dy, r.dz, r.tmin, r.tmax);
                        job.seed(sc, t);
                        active = true;
                    }
                }
                exhausted = base + (uint32_t)__popc(idle) >= n;
            }
        }
        if (!__any_sync(KZ_FULL, active)) break;
        int lost = 0;
#if KZ_TRAV_MODE == 1
        /* while-while: every lane descends until it holds triangles (or is finished), then the warp tests triangles together */
        while (active && !finished) {
            for (;;) {
                if (t.ng_y > 0x00FFFFFFu) kz_trav_node(sc, t, stk, ls);
                if (t.tg_y != 0u) break;
                if (t.ng_y <= 0x00FFFFFFu) {
                    if (t.sp == 0) break;
                    kz_trav_pop(t, stk, ls);
                }
            }
            while (t.tg_y != 0u) kz_trav_tri(sc, t);
            if (t.ng_y <= 0x00FFFFFFu) {
                if (t.sp == 0) finished = true;
                else kz_trav_pop(t, stk, ls);
            }
            if (!exhausted) {
                lost += 32 - __popc(__activemask()) - KZ_FETCH_ND;
                if (lost >= KZ_FETCH_NW) break;
            }
        }
#else
        while (active && !finished) {
#if KZ_WAIT_IDLE
            /* A lane whose triangles wait (too few lanes hold any) puts them on its stack only if it has a node group in hand to go
             * on with; otherwise it keeps them in registers and sits out the iteration -- pushing them would only be followed by
             * popping the same entry again (two entries each way, every iteration, until enough lanes have caught up). */
            if (t.tg_y == 0u && t.ng_y > 0x00FFFFFFu) kz_trav_node(sc, t, stk, ls);
            const int total = __popc(__activemask());
            while (t.tg_y != 0u) {
                if (__popc(__activemask()) * KZ_POSTPONE_DEN < total * KZ_POSTPONE_NUM) {
                    if (t.ng_y > 0x00FFFFFFu && t.sp < KZ_POSTPONE_SP_LIMIT) kz_trav_postpone(t, stk, ls);
                    break;
                }
                if (kz_trav_tri(sc, t) && Job::kStopsEarly && job.stop(sc, t)) { t.tg_y = 0u; t.ng_y = 0u; t.sp = 0; }
            }
            if (t.tg_y == 0u && t.ng_y <= 0x00FFFFFFu) {
                if (t.sp == 0) finished = true;
                else kz_trav_pop(t, stk, ls);
            }
#else
            if (t.ng_y > 0x00FFFFFFu) kz_trav_node(sc, t, stk, ls);
            const int total = __popc(__activemask());
            while (t.tg_y != 0u) {
                if (__popc(__activemask()) * KZ_POSTPONE_DEN < total * KZ_POSTPONE_NUM && t.sp < KZ_POSTPONE_SP_LIMIT) {   /* too few lanes have triangles: postpone */
                    kz_trav_postpone(t, stk, ls);
                    break;
                }
                if (kz_trav_tri(sc, t) && Job::kStopsEarly && job.stop(sc, t)) { t.tg_y = 0u; t.ng_y = 0u; t.sp = 0; }
            }
            if (t.ng_y <= 0x00FFFFFFu) {
                if (t.sp == 0) finished = true;
                else kz_trav_pop(t, stk, ls);
            }
#endif
            if (!exhausted) {
                lost += 32 - __popc(__activemask()) - KZ_FETCH_ND;
                if (lost >= KZ_FETCH_NW) break;
            }
        }
#endif
        __syncwarp();
    }
}

/* Append under divergence: the lanes that reach this call together are grouped by queue. */
__device__ __forceinline__ void kz_push_divergent(uint32_t *const *queues, uint32_t *counters, int which, uint32_t value) {
    const uint32_t peers = __match_any_sync(__activemask(), which);
    const uint32_t lane = kz_lane();
    const uint32_t leader = (uint32_t)__ffs((int)peers) - 1u;
    uint32_t base = 0u;
    if (lane == leader) base = atomicAdd(counters + which, (uint32_t)__popc(peers));
    base = __shfl_sync(peers, base, (int)leader);
    queues[which][base + (uint32_t)__popc(peers & ((1u << lane) - 1u))] = value;
}

/* Start of a chunk: raygen fills every slot, so the first extension pass takes slots 0 .. count-1 in order (k_extend<true> reads no queue). */
__global__ void k_chunk_reset(KzControl *ctl, uint32_t count, unsigned long long new_paths) {
    if (threadIdx.x == 0) {
        ctl->ext_shadow[0] = (unsigned long long)count; ctl->ext_shadow[1] = 0ull;
        ctl->paths += new_paths;
        for (int c = 0; c < KZ_NUM_CLASSES; ++c) ctl->n_class[c] = 0u;
        ctl->head_ext = ctl->head_shadow = ctl->head_trace = 0u;
    }
}
__global__ void k_bounce_reset(KzControl *ctl, int nxt) {
    if (threadIdx.x == 0) {
        ctl->ext_shadow[nxt] = 0ull;
        for (int c = 0; c < KZ_NUM_CLASSES; ++c) ctl->n_class[c] = 0u;
        ctl->head_ext = ctl->head_shadow = 0u;
    }
}

/* ---- raygen: renderer.cpp:20-33 + camera.cpp:70-91,191-223 ------------------------------- */
/* Slot i of the chunk = global path index first+i; a warp is one 8x4 pixel tile of one sample index: coherent primary rays,
 * and the splats of a warp land on neighbouring frame texels instead of piling onto one pixel.  Consecutive warps are
 * consecutive sample indices of the SAME tile (KzChunk::spp_group of them), so the warps resident on an SM walk the same
 * part of the accel and shade neighbouring surface points.
 * hint: per film pixel the (geomID, primID) its last primary ray hit, or nullptr (no hints).  With hints, raygen also runs the seed test
 * of the ray it has just generated against its pixel's hint (kz_seed_hit) and leaves the result, and the pixel, in the path's hit record
 * for k_extend<true>.  The test is a chain of dependent loads (hint, mesh, index record, vertices): here every lane of the warp runs it
 * at once, in a short kernel whose many resident warps hide the latency; at the refill point of the traversal loop only the refilled
 * lanes ran it while the whole warp waited. */
__global__ void __launch_bounds__(KZ_SHADE_THREADS) k_raygen(KzScene sc, KzPathState st, const uint2 *hint, KzChunk ch) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ch.count) return;
    /* path order: (block of spp_group sample indices, tile, sample index in the block, pixel of the tile) */
    unsigned long long g = ch.first + i;
    const unsigned long long per_block = (unsigned long long)ch.npx_padded * ch.spp_group;
    const uint32_t blk = (uint32_t)(g / per_block);
    g -= (unsigned long long)blk * per_block;
    const uint32_t left = ch.n_spp - blk * ch.spp_group;
    const uint32_t grp = left < ch.spp_group ? left : ch.spp_group;        /* the last block may be short */
    const uint32_t tile = (uint32_t)(g / (32u * grp));
    const uint32_t r = (uint32_t)(g - (unsigned long long)tile * (32u * grp));
    const uint32_t s_local = blk * ch.spp_group + (r >> 5), in_tile = r & 31u;
    const int x = ch.x0 + (int)((tile % ch.tiles_x) * 8u + (in_tile & 7u));
    const int y = ch.y0 + (int)((tile / ch.tiles_x) * 4u + (in_tile >> 3));
    KzHit seed; seed.t = seed.u = seed.v = 0.f; seed.prim = seed.geom = KZ_INVALID_ID;
    uint32_t pix = 0xFFFFFFFFu;
    if (x < ch.x1 && y < ch.y1) {
        const KzRayRec ray = kz_raygen_item(sc, st, i, x, y, (uint32_t)(ch.spp_begin + (int)s_local));
        if (hint != nullptr) {
            const uint2 h = hint[(size_t)y * (uint32_t)sc.camera.width + (uint32_t)x];
            kz_seed_hit(sc, ray.o.x, ray.o.y, ray.o.z, ray.d.x, ray.d.y, ray.d.z, ray.o.w, ray.d.w, h.x, h.y, seed);
            pix = (uint32_t)x | ((uint32_t)y << 16);
        }
    } else {
        /* padding lane of a tile that sticks out of the rectangle: a NaN ray (k_extend<true> drops it without counting it)
         * and the marker k_accumulate skips */
        const float nan = kz_u2f(0x7FC00000u);
        KzRayRec ray; ray.o = mkf4(0.f, 0.f, 0.f, 0.f); ray.d = mkf4(nan, nan, nan, 0.f);
        st.a[i].ray = ray;
        st.b[i].smp.pix = 0xFFFFFFFFu;
    }
    if (hint != nullptr) {
        KzHitRec rec = mk_hit_rec(seed);
        rec.pix = pix;
        st.a[i].hit = rec;
    }
}

/* ---- extend: Scene::rayIntersect for every queued path, then sort by material class ------- */
template <bool FIRST>
struct KzExtendJob {
    static constexpr bool kStopsEarly = false;
    __device__ __forceinline__ bool stop(const KzScene &, const KzTrav &) { return false; }
    const KzScene &sc; const KzPathState &st; KzControl *ctl; const KzQueues &q; const uint32_t *queue;
    uint2 *hint;                     /* primary rays: per film pixel the (geomID, primID) its last primary ray hit, or nullptr (no hints) */
    KzCounters cnt;
    uint32_t slot, n_seeded;
    KzHit first_hit; bool retraced;
    kz3 d;
    __device__ KzExtendJob(const KzScene &s, const KzPathState &p, KzControl *c, const KzQueues &qq, const uint32_t *qu, uint2 *h)
        : sc(s), st(p), ctl(c), q(qq), queue(qu), hint(h), n_seeded(0u) { cnt.paths = cnt.rays_ext = cnt.rays_shadow = cnt.vertices = cnt.rays_seeded = 0ull; }
    /* hint slot of the path's pixel (KzHitRec::pix, written by k_raygen); ~0 for its padding lanes (0xFFFFFFFF lies outside every film) */
    __device__ __forceinline__ size_t hint_index() const {
        const uint32_t pix = st.a[slot].hit.pix, px = pix & 0xFFFFu, py = pix >> 16;
        if (px >= (uint32_t)sc.camera.width || py >= (uint32_t)sc.camera.height) return ~(size_t)0;
        return (size_t)py * (uint32_t)sc.camera.width + px;
    }
    /* One triangle covers several pixels and every pixel is sampled many times, so the triangle the pixel's last primary ray hit is
     * usually hit again: as the preset best hit it lets the node step cull with its t from the root on, instead of walking every
     * box along the ray up to the hit.  The hit found is the same either way (kz_seed_hit).  k_raygen ran the seed test; this loads its
     * result (one load: the slot is the item) and installs it.  Loaded here rather than with the ray in begin(), it is not held across
     * kz_trav_init: 52 instead of 72 bytes of spills. */
    __device__ __forceinline__ void seed(const KzScene &, KzTrav &t) {
        if (!FIRST || hint == nullptr) return;
        const KzHitRec s = st.a[slot].hit;
        KzHit h; h.t = s.t; h.u = s.u; h.v = s.v; h.prim = s.prim; h.geom = s.geom;
        n_seeded += kz_trav_preset(t, h) ? 1u : 0u;
    }
    __device__ __forceinline__ void begin(uint32_t item, KzRayIn &r) {
        slot = FIRST ? item : queue[item];          /* the first pass takes the chunk's slots in order (k_chunk_reset) */
        const KzRayRec ray = st.a[slot].ray;
        const KzF4 ro = ray.o, rd = ray.d;
        r.ox = ro.x; r.oy = ro.y; r.oz = ro.z; r.tmin = ro.w; r.dx = rd.x; r.dy = rd.y; r.dz = rd.z; r.tmax = rd.w;
        d = mk3(rd.x, rd.y, rd.z);
        retraced = false;
    }
    __device__ __forceinline__ bool end(uint32_t, const KzHit &hit, KzRayIn &r) {
        if (FIRST && isnan(d.x)) return false;          /* padding slot of k_raygen: not a path */
        cnt.rays_ext += 1;
        KzHit h = hit;
        if (FIRST) {
            /* the hint for the pixel's next sample: what this first trace hit (a miss clears it).  Samples of one pixel in flight
             * together race on the slot; whichever store lands, it is a triangle (or none) and only ever a hint. */
            if (hint != nullptr && !retraced) { const size_t i = hint_index(); if (i != ~(size_t)0) hint[i] = make_uint2(h.geom, h.prim); }
            if (retraced) { if (h.geom == KZ_INVALID_ID) h = first_hit; }     /* a miss keeps the light hit */
            else if (h.geom != KZ_INVALID_ID && sc.integrator.type == KZ_INTEGRATOR_PATH_MIS) {
                const uint32_t fl = sc.meshes[h.geom].flags;
                if ((fl & KZ_MESH_IS_LIGHT) && !(fl & KZ_MESH_LIGHT_VISIBLE)) {
                    /* integrator.cpp:214-219: one re-trace from its.p + eps*d with a default Ray3f */
                    KzIts its; its.acc_rough = 0.f;
                    fill_intersection(sc, h, its, mk3(0.f));
                    const kz3 o = its.p + sc.integrator.trace_bias * d;
                    r.ox = o.x; r.oy = o.y; r.oz = o.z; r.tmin = KZ_EPSILON; r.dx = d.x; r.dy = d.y; r.dz = d.z; r.tmax = KZ_INF;
                    first_hit = h; retraced = true;
                    return true;
                }
            }
        }
        st.a[slot].hit = mk_hit_rec(h);
        kz_push_divergent(q.cls, ctl->n_class, kz_classify(sc, h.geom), slot);
        return false;
    }
};

/* hint: k_extend<true> only (primary rays), nullptr = no hints */
template <bool FIRST>
__global__ void __launch_bounds__(KZ_TRACE_THREADS, KZ_TRACE_MIN_BLOCKS) k_extend(KzScene sc, KzPathState st, KzControl *ctl, KzQueues q, int cur, uint2 *hint) {
    const KzStackRef stk = kz_trav_shared_init();
    KzExtendJob<FIRST> job(sc, st, ctl, q, q.ext[cur], FIRST ? hint : nullptr);
    kz_warp_trace(sc, stk, &ctl->head_ext, kz_ext_count(ctl, cur), job);
    job.cnt.rays_seeded = job.n_seeded;
    kz_flush_counters(ctl, job.cnt);
}

/* ---- shade: one integrator loop iteration for every path of one material class ------------ */
#ifndef KZ_SHADE_BLOCK_PUSH
#define KZ_SHADE_BLOCK_PUSH 1
#endif
#ifndef KZ_SHADE_MIN_BLOCKS_DIFFUSE
#define KZ_SHADE_MIN_BLOCKS_DIFFUSE 8       /* 64 registers: measured 4 -> 1038, 5 -> 1060, 6 -> 1056, 8 -> 1077 Mpaths/s */
#endif
#ifndef KZ_SHADE_MIN_BLOCKS_TERMINAL
#define KZ_SHADE_MIN_BLOCKS_TERMINAL 4
#endif
#ifndef KZ_SHADE_MIN_BLOCKS
#define KZ_SHADE_MIN_BLOCKS 4
#endif
template <int CLS>
__global__ void __launch_bounds__(KZ_SHADE_THREADS, (CLS == KZ_CLASS_DIFFUSE ? KZ_SHADE_MIN_BLOCKS_DIFFUSE : (CLS == KZ_CLASS_TERMINAL ? KZ_SHADE_MIN_BLOCKS_TERMINAL : KZ_SHADE_MIN_BLOCKS))) k_shade(KzScene sc, KzPathState st, KzControl *ctl, KzQueues q, int nxt, int bounce) {
    const uint32_t n = ctl->n_class[CLS];
    const uint32_t *queue = q.cls[CLS];
    const uint32_t stride = gridDim.x * blockDim.x;
    KzCounters cnt; cnt.paths = cnt.rays_ext = cnt.rays_shadow = cnt.vertices = cnt.rays_seeded = 0ull;
#if KZ_SHADE_BLOCK_PUSH
    /* queue space for the whole CTA with ONE packed atomic per iteration (the counter is a single address: 1.8 M warp-level
     * atomics per frame serialise in the L2) */
    constexpr int NW = KZ_SHADE_THREADS / 32;
    __shared__ uint32_t s_cnt[2][2][NW];
    __shared__ unsigned long long s_base[2];
    int par = 0;
    for (uint32_t bbase = blockIdx.x * blockDim.x; bbase < n; bbase += stride, par ^= 1) {
        const uint32_t idx = bbase + threadIdx.x;
        uint32_t slot = 0u, flags = 0u;
        if (idx < n) {
            slot = queue[idx];
            flags = kz_shade_item<CLS>(sc, st, slot, bounce, cnt);
        }
        if (CLS != KZ_CLASS_TERMINAL) {
            const bool pa = (flags & KZ_SHADE_CONTINUE) != 0u, pb = (flags & KZ_SHADE_SHADOW) != 0u;
            const uint32_t ma = __ballot_sync(KZ_FULL, pa), mb = __ballot_sync(KZ_FULL, pb);
            const uint32_t w = threadIdx.x >> 5, lane = kz_lane(), lt = (1u << lane) - 1u;
            if (lane == 0u) { s_cnt[par][0][w] = (uint32_t)__popc(ma); s_cnt[par][1][w] = (uint32_t)__popc(mb); }
            __syncthreads();
            if (threadIdx.x == 0) {
                uint32_t ta = 0u, tb = 0u;
#pragma unroll
                for (int k = 0; k < NW; ++k) { ta += s_cnt[par][0][k]; tb += s_cnt[par][1][k]; }
                s_base[par] = (ta | tb) ? atomicAdd(&ctl->ext_shadow[nxt], (unsigned long long)ta | ((unsigned long long)tb << 32)) : 0ull;
            }
            __syncthreads();
            uint32_t oa = (uint32_t)(s_base[par] & 0xFFFFFFFFull), ob = (uint32_t)(s_base[par] >> 32);
#pragma unroll
            for (int k = 0; k < NW; ++k) if ((uint32_t)k < w) { oa += s_cnt[par][0][k]; ob += s_cnt[par][1][k]; }
            if (pa) q.ext[nxt][oa + (uint32_t)__popc(ma & lt)] = slot;
            if (pb) q.shadow[ob + (uint32_t)__popc(mb & lt)] = slot;
        }
    }
#else
    for (uint32_t base = (blockIdx.x * blockDim.x + threadIdx.x) & ~31u; base < n; base += stride) {
        const uint32_t idx = base + kz_lane();
        uint32_t slot = 0u, flags = 0u;
        if (idx < n) {
            slot = queue[idx];
            flags = kz_shade_item<CLS>(sc, st, slot, bounce, cnt);
        }
        __syncwarp();
        if (CLS != KZ_CLASS_TERMINAL)
            kz_push2(q.ext[nxt], q.shadow, &ctl->ext_shadow[nxt], (flags & KZ_SHADE_CONTINUE) != 0u, (flags & KZ_SHADE_SHADOW) != 0u, slot);
    }
#endif
    kz_flush_counters(ctl, cnt);
}

/* ---- shadow: integrator.cpp:259-294 ------------------------------------------------------- */
/* The closest-hit walk through invisible lights (kz_occluded_walk) as a job: every segment is one ray. */
struct KzWalk {
    kz3 o, d; float tmax; int seg;
    __device__ __forceinline__ void start(KzRayIn &r, kz3 o_, kz3 d_, float tmin, float tmax_) {
        o = o_; d = d_; tmax = tmax_; seg = 0;
        r.ox = o.x; r.oy = o.y; r.oz = o.z; r.tmin = tmin; r.dx = d.x; r.dy = d.y; r.dz = d.z; r.tmax = tmax;
    }
    /* The walk only asks whether its ray reaches something opaque.  A hit on an opaque mesh settles that as soon as no invisible
     * emitter can lie in front of it -- none in the scene, or the ray up to the hit stays outside their bounds: the closest hit of
     * this segment is then opaque too, whichever triangle it is, and step() answers "occluded" exactly as for the closest one. */
    __device__ __forceinline__ static bool settles(const KzScene &sc, const KzTrav &t) {
        if (sc.integrator.type != KZ_INTEGRATOR_PATH_MIS) return true;                      /* ao / whitted: any hit occludes */
        const uint32_t fl = sc.meshes[t.best.geom].flags;
        if ((fl & KZ_MESH_IS_LIGHT) && !(fl & KZ_MESH_LIGHT_VISIBLE)) return false;
        return sc.n_invisible_lights == 0 || kz_trav_misses_box(t, sc.inv_light_lo, sc.inv_light_hi, t.best.t);
    }
    /* returns 0 = unoccluded, 1 = occluded, 2 = continue with the ray written to r */
    __device__ __forceinline__ int step(const KzScene &sc, const KzHit &h, float eps, KzRayIn &r) {
        ++seg;
        if (h.geom == KZ_INVALID_ID) return 0;
        const uint32_t fl = sc.meshes[h.geom].flags;
        if (!(fl & KZ_MESH_IS_LIGHT) || (fl & KZ_MESH_LIGHT_VISIBLE) || sc.integrator.type != KZ_INTEGRATOR_PATH_MIS) return 1;     /* ao / whitted: any hit occludes */
        if (seg > 4096) return 0;
        o = o + d * (h.t + eps);
        tmax = tmax - h.t;
        r.ox = o.x; r.oy = o.y; r.oz = o.z; r.tmin = eps; r.dx = d.x; r.dy = d.y; r.dz = d.z; r.tmax = tmax;
        return 2;
    }
};
struct KzShadowJob {
    static constexpr bool kStopsEarly = true;
    __device__ __forceinline__ bool stop(const KzScene &s, const KzTrav &t) { return KzWalk::settles(s, t); }
    __device__ __forceinline__ void seed(const KzScene &, KzTrav &) {}
    const KzScene &sc; const KzPathState &st; const uint32_t *queue;
    KzCounters cnt; uint32_t slot; KzWalk walk;
    __device__ KzShadowJob(const KzScene &s, const KzPathState &p, const uint32_t *qu) : sc(s), st(p), queue(qu) { cnt.paths = cnt.rays_ext = cnt.rays_shadow = cnt.vertices = cnt.rays_seeded = 0ull; }
    __device__ __forceinline__ void begin(uint32_t item, KzRayIn &r) {
        slot = queue[item];
        const KzF4 so = st.a[slot].ray.o;
        const KzShdRec shd = st.c[slot].shd;
        walk.start(r, mk3(so.x, so.y, so.z), mk3(shd.d.x, shd.d.y, shd.d.z), shd.pending.w, shd.d.w);
    }
    __device__ __forceinline__ bool end(uint32_t, const KzHit &h, KzRayIn &r) {
        cnt.rays_shadow += 1;
        const int s = walk.step(sc, h, sc.integrator.trace_bias, r);
        if (s == 2) return true;
        if (s == 0) {
            const KzF4 p = st.c[slot].shd.pending;
            KzF4 L = st.b[slot].rad.L;
            L.x += p.x; L.y += p.y; L.z += p.z;
            st.b[slot].rad.L = L;
        }
        return false;
    }
};
__global__ void __launch_bounds__(KZ_TRACE_THREADS, KZ_TRACE_MIN_BLOCKS) k_shadow(KzScene sc, KzPathState st, KzControl *ctl, KzQueues q, int nxt) {
    const KzStackRef stk = kz_trav_shared_init();
    KzShadowJob job(sc, st, q.shadow);
    kz_warp_trace(sc, stk, &ctl->head_shadow, kz_shadow_count(ctl, nxt), job);
    kz_flush_counters(ctl, job.cnt);
}

/* ---- accumulate: ImageBlock::put over the whole chunk (block.cpp:56-85) ------------------- */
#ifndef KZ_ACC_MAX_TEXELS
#define KZ_ACC_MAX_TEXELS 160        /* (8 + span) x (4 + span) texels of a tile's footprint region: span 4 (radius 2) -> 96, span 6 -> 140 */
#endif
/* Every warp splats its own run of consecutive 32-path units.  In path order the next units are the same 8x4-pixel tile's next sample
 * indices, whose splats land on the same (8 + span) x (4 + span) frame texels: the warp sums them in shared memory and adds the region
 * to the frame once per tile -- 3 global reductions per lane and tile instead of 16-25 per path.  No shared-memory atomics are needed:
 * the taps are walked by their offset from the path's own pixel, and at a given offset the 32 paths of a unit (32 different pixels)
 * touch 32 different texels.  (rx0, ry0): origin of the request rectangle, which the tiles are aligned to. */
__global__ void __launch_bounds__(KZ_SHADE_THREADS) k_accumulate(KzScene sc, KzPathState st, uint32_t count, KzF4 *frame, int rx0, int ry0) {
    __shared__ float s_table[33];
    __shared__ KzF4 s_region[KZ_SHADE_THREADS / 32][KZ_ACC_MAX_TEXELS];
    if (threadIdx.x < 33) s_table[threadIdx.x] = sc.filter.table[threadIdx.x];
    const uint32_t lane = threadIdx.x & 31u;
    KzF4 *region = s_region[threadIdx.x >> 5];
    for (uint32_t e = lane; e < KZ_ACC_MAX_TEXELS; e += 32u) region[e] = mkf4(0.f, 0.f, 0.f, 0.f);
    __syncthreads();
    const float radius = sc.filter.radius, lookup = 32 / radius;
    const int b = sc.border, cols = sc.camera.width + 2 * b, rows = sc.camera.height + 2 * b;
    const int lo = -(int)floorf(radius + 0.5f), hi = (int)ceilf(radius + 0.5f) - 1;      /* tap offsets from the path's own pixel */
    const int tw = 8 + hi - lo, th = 4 + hi - lo;
    const bool tiled = tw * th <= KZ_ACC_MAX_TEXELS;
    const uint32_t n_units = (count + 31u) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, per = (n_units + n_warps - 1u) / n_warps;
    const uint32_t u1 = min(n_units, (w + 1u) * per);
    int cur_x = 0, cur_y = 0; bool open = false;          /* tile whose sums the region holds */
    for (uint32_t u = w * per; u < u1; ++u) {
        const uint32_t i = (u << 5) + lane;
        KzSplat sp = {};
        bool ok = i < count && st.b[i].smp.pix != 0xFFFFFFFFu && kz_splat_of(sc, st, i, sp);
        if (!tiled) { if (ok) kz_accumulate_item(sc, st, i, frame, s_table); continue; }
        /* a footprint that does not fit the offsets walked below (it always does for sample positions in [0, 1)) goes the direct way */
        if (ok && (sp.x0 < sp.ipx + b + lo || sp.x1 > sp.ipx + b + hi || sp.y0 < sp.ipy + b + lo || sp.y1 > sp.ipy + b + hi)) { kz_accumulate_item(sc, st, i, frame, s_table); ok = false; }
        const uint32_t m = __ballot_sync(KZ_FULL, ok);
        if (!m) continue;
        const int leader = __ffs((int)m) - 1;
        const int tx = __shfl_sync(KZ_FULL, ok ? rx0 + ((sp.ipx - rx0) & ~7) : 0, leader), ty = __shfl_sync(KZ_FULL, ok ? ry0 + ((sp.ipy - ry0) & ~3) : 0, leader);
        if (open && (tx != cur_x || ty != cur_y)) {       /* next tile: hand the finished one to the frame */
            for (int e = (int)lane; e < tw * th; e += 32) {
                const KzF4 v = region[e];
                const int X = cur_x + b + lo + e % tw, Y = cur_y + b + lo + e / tw;
                if ((v.x != 0.f || v.y != 0.f || v.z != 0.f || v.w != 0.f) && X >= 0 && X < cols && Y >= 0 && Y < rows) KZ_FRAME_ADD(frame + ((size_t)Y * cols + X), v.x, v.y, v.z, v.w);
                region[e] = mkf4(0.f, 0.f, 0.f, 0.f);
            }
            __syncwarp();
        }
        cur_x = tx; cur_y = ty; open = true;
        const int bx = ok ? sp.ipx - tx - lo : 0, by = ok ? sp.ipy - ty - lo : 0;      /* region column / row of the tap at offset (lo, lo) */
        for (int dy = lo; dy <= hi; ++dy) {
            const int Y = sp.ipy + b + dy;
            const bool rowok = ok && Y >= sp.y0 && Y <= sp.y1;
            const float wy = rowok ? s_table[(int)(fabsf((float)Y - sp.py) * lookup)] : 0.f;
            for (int dx = lo; dx <= hi; ++dx) {
                const int X = sp.ipx + b + dx;
                if (rowok && X >= sp.x0 && X <= sp.x1) {
                    const float wx = s_table[(int)(fabsf((float)X - sp.px) * lookup)];
                    KzF4 *p = region + ((by + dy) * tw + (bx + dx));
                    KzF4 v = *p;
                    v.x += sp.value.x * wx * wy; v.y += sp.value.y * wx * wy; v.z += sp.value.z * wx * wy; v.w += 1.0f * wx * wy;
                    *p = v;
                }
                __syncwarp();
            }
        }
    }
    if (tiled && open) {
        __syncwarp();
        for (int e = (int)lane; e < tw * th; e += 32) {
            const KzF4 v = region[e];
            const int X = cur_x + b + lo + e % tw, Y = cur_y + b + lo + e / tw;
            if ((v.x != 0.f || v.y != 0.f || v.z != 0.f || v.w != 0.f) && X >= 0 && X < cols && Y >= 0 && Y < rows) KZ_FRAME_ADD(frame + ((size_t)Y * cols + X), v.x, v.y, v.z, v.w);
        }
    }
}

/* ---- batch entry points (parity tests + intersection microbench) -------------------------- */
/* kzgpu_trace: rays/hits in the C-ABI's AoS layout (32 B in, 20 B out). */
struct KzTraceJob {
    static constexpr bool kStopsEarly = false;
    __device__ __forceinline__ bool stop(const KzScene &, const KzTrav &) { return false; }
    __device__ __forceinline__ void seed(const KzScene &, KzTrav &) {}
    const KzF4 *rays; float *hits;
    __device__ __forceinline__ void begin(uint32_t item, KzRayIn &r) {
        const KzU4 a = kz_load_u4(rays + 2 * (size_t)item), b = kz_load_u4(rays + 2 * (size_t)item + 1);
        r.ox = kz_u2f(a.x); r.oy = kz_u2f(a.y); r.oz = kz_u2f(a.z); r.tmin = kz_u2f(a.w);
        r.dx = kz_u2f(b.x); r.dy = kz_u2f(b.y); r.dz = kz_u2f(b.z); r.tmax = kz_u2f(b.w);
    }
    __device__ __forceinline__ bool end(uint32_t item, const KzHit &h, KzRayIn &) {
        float *o = hits + 5 * (size_t)item;
        o[0] = h.t; o[1] = h.u; o[2] = h.v; o[3] = kz_u2f(h.prim); o[4] = kz_u2f(h.geom);
        return false;
    }
};
__global__ void __launch_bounds__(KZ_TRACE_THREADS, KZ_BATCH_MIN_BLOCKS) k_trace(KzScene sc, const KzF4 *rays, uint32_t n, float *hits, uint32_t *cursor, KzControl *ctl) {
    const KzStackRef stk = kz_trav_shared_init();
    KzTraceJob job; job.rays = rays; job.hits = hits;
    kz_warp_trace(sc, stk, cursor, n, job);
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&ctl->rays_ext, (unsigned long long)n);
}

struct KzOccludedJob {
    static constexpr bool kStopsEarly = true;
    __device__ __forceinline__ bool stop(const KzScene &s, const KzTrav &t) { return KzWalk::settles(s, t); }
    __device__ __forceinline__ void seed(const KzScene &, KzTrav &) {}
    const KzScene &sc; const KzF4 *rays; float eps; uint8_t *occ, *segments;
    KzCounters cnt; KzWalk walk;
    __device__ KzOccludedJob(const KzScene &s, const KzF4 *r, float e, uint8_t *o, uint8_t *sg) : sc(s), rays(r), eps(e), occ(o), segments(sg) {
        cnt.paths = cnt.rays_ext = cnt.rays_shadow = cnt.vertices = cnt.rays_seeded = 0ull;
    }
    __device__ __forceinline__ void begin(uint32_t item, KzRayIn &r) {
        const KzU4 a = kz_load_u4(rays + 2 * (size_t)item), b = kz_load_u4(rays + 2 * (size_t)item + 1);
        walk.start(r, mk3(kz_u2f(a.x), kz_u2f(a.y), kz_u2f(a.z)), mk3(kz_u2f(b.x), kz_u2f(b.y), kz_u2f(b.z)), kz_u2f(a.w), kz_u2f(b.w));
    }
    __device__ __forceinline__ bool end(uint32_t item, const KzHit &h, KzRayIn &r) {
        cnt.rays_shadow += 1;
        const int s = walk.step(sc, h, eps, r);
        if (s == 2) return true;
        occ[item] = (uint8_t)s;
        if (segments) segments[item] = (uint8_t)(walk.seg > 255 ? 255 : walk.seg);
        return false;
    }
};
__global__ void __launch_bounds__(KZ_TRACE_THREADS, KZ_BATCH_MIN_BLOCKS) k_occluded(KzScene sc, const KzF4 *rays, uint32_t n, float eps, uint8_t *occ, uint8_t *segments,
                                                                uint32_t *cursor, KzControl *ctl) {
    const KzStackRef stk = kz_trav_shared_init();
    KzOccludedJob job(sc, rays, eps, occ, segments);
    kz_warp_trace(sc, stk, cursor, n, job);
    kz_flush_counters(ctl, job.cnt);
}

/* kzgpu_sample_dump: sampler.cpp generateSample + draw pattern, one thread per (pixel, sample) */
__global__ void k_sample_dump(KzScene sc, const int32_t *triples, uint32_t n, const char *pattern, uint32_t per, float *out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    KzSampler sm;
    kz_sampler_start(sc, sm, triples[3 * i], triples[3 * i + 1], (uint32_t)triples[3 * i + 2]);
    float *o = out + (size_t)i * per;
    for (const char *p = pattern; *p; ++p) {
        if (*p == '1') *o++ = kz_next1d(sc, sm);
        else { const kz2 v = (*p == 'P') ? kz_next_pixel2d(sc, sm) : kz_next2d(sc, sm); *o++ = v.x; *o++ = v.y; }
    }
}

__global__ void k_camera_rays(KzScene sc, const KzF4 *samples, uint32_t n, KzF4 *out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const KzF4 s = samples[i];
    KzF4 ro, rd;
    kz_camera_ray(sc.camera, mk2(s.x, s.y), mk2(s.z, s.w), ro, rd);
    out[2 * (size_t)i] = ro; out[2 * (size_t)i + 1] = rd;
}

/* One BSDF query per thread in an identity shading frame (parity of the shading library). */
struct KzBsdfQuery { float wi[3], wo[3], uv[2], acc_rough, s1, s2[2]; int32_t mesh, mode; };
__global__ void k_bsdf_query(KzScene sc, const KzBsdfQuery *qs, uint32_t n, float *out8) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const KzBsdfQuery q = qs[i];
    KzIts its;
    its.sh.s = mk3(1, 0, 0); its.sh.t = mk3(0, 1, 0); its.sh.n = mk3(0, 0, 1);
    its.geo_n = its.sh.n; its.dpdu = mk3(1, 0, 0); its.uv = mk2(q.uv[0], q.uv[1]); its.mesh = q.mesh; its.acc_rough = q.acc_rough;
    its.p = mk3(0.f);
    const KzBsdfCtx bc = bsdf_ctx(sc, its);
    float *o = out8 + 8 * (size_t)i;
    for (int k = 0; k < 8; ++k) o[k] = 0.f;
    const kz3 wi = mk3(q.wi[0], q.wi[1], q.wi[2]);
    if (q.mode == 2) {
        kz3 w_o; float pdf, eta_s; int measure;
        const kz3 w = bsdf_sample(bc, its, wi, q.s1, mk2(q.s2[0], q.s2[1]), &w_o, &pdf, &measure, &eta_s);
        o[0] = w.x; o[1] = w.y; o[2] = w.z;
        if (!iszero(w)) { o[3] = w_o.x; o[4] = w_o.y; o[5] = w_o.z; o[7] = pdf; }
        o[6] = (float)measure;
        return;
    }
    kz3 f; float pdf;
    bsdf_eval_pdf(bc, its, wi, mk3(q.wo[0], q.wo[1], q.wo[2]), &f, &pdf);
    if (q.mode == 0) { o[0] = f.x; o[1] = f.y; o[2] = f.z; } else o[0] = pdf;
}

/* ---- textures: mip pyramid build + lookup probe ----------------------------------------- */
__global__ void k_mip_level(KzF4 *texels, size_t src_off, int sw, int sh, size_t dst_off, int dw, int dh) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= dw || y >= dh) return;
    const int x0 = min(2 * x, sw - 1), x1 = min(2 * x + 1, sw - 1), y0 = min(2 * y, sh - 1), y1 = min(2 * y + 1, sh - 1);
    const KzF4 a = texels[src_off + (size_t)y0 * sw + x0], b = texels[src_off + (size_t)y0 * sw + x1];
    const KzF4 c = texels[src_off + (size_t)y1 * sw + x0], d = texels[src_off + (size_t)y1 * sw + x1];
    KzF4 r; r.x = 0.25f * (a.x + b.x + c.x + d.x); r.y = 0.25f * (a.y + b.y + c.y + d.y); r.z = 0.25f * (a.z + b.z + c.z + d.z); r.w = 1.f;
    texels[dst_off + (size_t)y * dw + x] = r;
}
__global__ void k_image_lookup(KzScene sc, int image, int level, const float *st, uint32_t n, float *rgb) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const kz3 c = kz_image_bicubic(sc, image, st[2 * i], st[2 * i + 1], level);
    rgb[3 * i] = c.x; rgb[3 * i + 1] = c.y; rgb[3 * i + 2] = c.z;
}

/* ---- resolve: block.cpp:39-45 + common.cpp:352-366 + bitmap.cpp:46-54 --------------------- */
__global__ void k_resolve(const KzF4 *frame, int width, int height, int border, float *rgb, uint8_t *srgb8) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= width || y >= height) return;
    const KzF4 v = frame[(size_t)(y + border) * (width + 2 * border) + (x + border)];
    kz3 c = v.w != 0.f ? mk3(v.x / v.w, v.y / v.w, v.z / v.w) : mk3(0.f);
    const size_t o = 3 * ((size_t)y * width + x);
    if (rgb) { rgb[o] = c.x; rgb[o + 1] = c.y; rgb[o + 2] = c.z; }
    if (srgb8) {
        const float s[3] = {linear_to_srgb1(c.x), linear_to_srgb1(c.y), linear_to_srgb1(c.z)};
        for (int k = 0; k < 3; ++k) srgb8[o + k] = (uint8_t)clampf(255.f * s[k], 0.f, 255.f);
    }
}

/* ---- parity probes: post-intersection record and emitter sample, field by field --------------------------------------- */
/* accel.cpp:63-236 for one ray per thread (plain per-ray loop; this is a probe, not a hot path) */
__global__ void __launch_bounds__(KZ_TRACE_THREADS) k_intersection_dump(KzScene sc, const KzF4 *rays, uint32_t n, float *out24) {
    const KzStackRef stk = kz_trav_shared_init();
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const KzF4 ro = rays[2 * (size_t)i], rd = rays[2 * (size_t)i + 1];
    const KzHit h = kz_trace(sc, stk, ro.x, ro.y, ro.z, rd.x, rd.y, rd.z, ro.w, rd.w, false);
    float *o = out24 + 24 * (size_t)i;
    for (int k = 0; k < 24; ++k) o[k] = 0.f;
    o[0] = h.t; o[1] = -1.f;
    if (h.geom == KZ_INVALID_ID) return;
    KzIts its; its.acc_rough = 0.f;
    fill_intersection(sc, h, its, mk3(0.f));
    o[1] = (float)its.mesh;
    o[2] = its.p.x; o[3] = its.p.y; o[4] = its.p.z; o[5] = its.uv.x; o[6] = its.uv.y;
    o[7] = its.geo_n.x; o[8] = its.geo_n.y; o[9] = its.geo_n.z;
    o[10] = its.sh.s.x; o[11] = its.sh.s.y; o[12] = its.sh.s.z;
    o[13] = its.sh.t.x; o[14] = its.sh.t.y; o[15] = its.sh.t.z;
    o[16] = its.sh.n.x; o[17] = its.sh.n.y; o[18] = its.sh.n.z;
    o[19] = its.dpdu.x; o[20] = its.dpdu.y; o[21] = its.dpdu.z;
}

/* scene.h:45-56 + mesh.cpp:108-133 + light.cpp:16-51 */
__global__ void k_light_sample_dump(KzScene sc, const float *ref3, const float *u5, uint32_t n, float *out16) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float *o = out16 + 16 * (size_t)i;
    for (int k = 0; k < 16; ++k) o[k] = 0.f;
    o[0] = -1.f;
    if (sc.n_light_meshes <= 0) return;
    const float *u = u5 + 5 * (size_t)i;
    const KzEmitterSample es = kz_sample_emitter(sc, mk3(ref3[3 * (size_t)i], ref3[3 * (size_t)i + 1], ref3[3 * (size_t)i + 2]), u[0], u[1], u[2], u[3]);
    o[0] = (float)es.mesh;
    o[1] = es.p.x; o[2] = es.p.y; o[3] = es.p.z; o[4] = es.n.x; o[5] = es.n.y; o[6] = es.n.z;
    o[7] = es.wi.x; o[8] = es.wi.y; o[9] = es.wi.z; o[10] = es.dist; o[11] = es.pdf;
    if (es.pdf > 0.f && !isnan(es.pdf) && !isinf(es.pdf)) {
        const kz_light_desc l = sc.lights[es.light];
        const kz3 Ls = mk3(l.radiance[0], l.radiance[1], l.radiance[2]) / es.pdf;
        o[12] = Ls.x; o[13] = Ls.y; o[14] = Ls.z;
    }
}

#endif
