// context.hpp — host-side state of one trace_ctx (one GPU, one stream) shared by the .cu translation units.
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <string>
#include <vector>

#include "device_common.cuh"

// NVTX ranges around the wavefront stages (SURVEY.md §5): header-only NVTX3, a no-op unless a profiler is attached
#if defined(__has_include)
#if __has_include(<nvtx3/nvToolsExt.h>)
#include <nvtx3/nvToolsExt.h>
#define TR_HAVE_NVTX 1
#endif
#endif
struct TrRange {
#ifdef TR_HAVE_NVTX
    explicit TrRange(const char* name) { nvtxRangePushA(name); }
    ~TrRange() { nvtxRangePop(); }
#else
    explicit TrRange(const char*) {}
#endif
    TrRange(const TrRange&) = delete;
    TrRange& operator=(const TrRange&) = delete;
};

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    // grow-only device allocation
    cudaError_t ensure(size_t need) {
        if (need <= bytes) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; bytes = 0;
        size_t want = need + need / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) bytes = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct SppmState;

struct trace_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    // lanes: independent sub-batches of a render run concurrently on side streams (each with its own queues and
    // counter block) so that one lane's latency-bound deep-bounce launches overlap another lane's wide ones
    static const int MAX_LANES = 16;
    cudaStream_t side[MAX_LANES] = {};
    cudaEvent_t ev_fork = nullptr, ev_join[MAX_LANES] = {};
    // the serial chain of an SPPM iteration (grid -> deposits -> all-reduce -> update) runs on a stream of the greatest
    // priority: its launches overtake the run-ahead camera / photon launches of later iterations when CTA slots free up
    cudaStream_t chain_stream = nullptr;
    cudaStream_t coll_stream = nullptr;     // SPPM collectives (same priority): the next all-gather overlaps this iteration's chain
    cudaEvent_t ev_chain = nullptr;
    int sppm_chain_priority = 1;            // option: 0 keeps the chain on the caller's stream
    cudaStream_t copy_stream = nullptr;     // host film upload of trace_render_whitted, overlapped with the render
    cudaEvent_t ev_copy = nullptr;
    bool film_upload_pending = false;       // the film merge must wait for ev_copy
    cudaStream_t cur_stream = nullptr;      // stream the launch helpers enqueue on (== stream outside a laned render)
    int cur_lane = 0;
    int lanes = 12;
    int num_sms = 148;
    std::string err;

    // options
    int slab = 2;                 // 0 literal reference slab test, 1 textbook (not hit-equivalent), 2 guarded (default)
    int64_t batch = 1 << 26;      // camera samples per wavefront batch (queues: ~350 B per sample, allocated for min(batch, work))
    int count_nodes = 0;
    int cap_percent = 200;        // ray-queue capacity per bounce level, in % of the batch size
    int persist = 0;              // dynamic ray fetch in the traversal kernels: 0 off, 1 bounce levels >= 2 and shadow rays, 2 all
    int sppm_path = 0;            // SPPM: bounce levels the fused path kernel carries before handing over to the wavefront queues (0: none)
    int fuse_primary = 1;         // Whitted: generate + trace the camera rays in one kernel (no primary-ray queue)
    int cur_level = 0;            // bounce level of the extend launch being enqueued (set by the integrators)
    int work_slot = 0;
    int leaf_wait = -1;           // walk selector: -1 pair nodes (default, option "walk" 1), 0 the reference loop ("walk" 0), 4/8/16/32 batched leaves
    int time_kernels = 0;
    int shadow_tree = 1;          // any-hit queries walk the scene's shadow tree (traverse_shadow) when it has one; 0 = the reference tree only
    int rank = 0, world = 1;
    void* comm = nullptr;         // ncclComm_t of this rank (comm.cpp), null until trace_comm_init
    int nccl_version = 0;
    // Peer-memory film sum (whitted.cu k_film_sum_p2p, comm.cpp comm_p2p_exchange): every rank's private film lives in an
    // allocation the other ranks map (CUDA IPC between processes, plain peer access between threads of one process); the
    // merge kernel of a rank then reads its band of ALL films over NVLink, sums and merges in one pass - no NCCL ring.
    int film_p2p = 1;             // option: 0 = NCCL collectives only
    DevBuf p2p_film;              // [private film | summed film (film_mode 0: the bands land in rank 0's)]
    size_t p2p_npix = 0;          // padded pixel count the peers' mappings were exchanged for
    int p2p_state = 0;            // 1 usable, -1 tried and failed on some rank (NCCL path), 0 not tried for this size
    std::vector<void*> p2p_peer;  // rank r's p2p_film base in this process's address space
    std::vector<void*> p2p_opened;   // IPC mappings to close
    int film_sum = 0;             // film_mode 0: 0 = ncclReduce to rank 0, 1 = ncclAllReduce, 2 = reduce-scatter + gather of the chunks onto rank 0
    int film_mode = 0;            // multi-rank Whitted film delivery: 0 = whole film summed onto rank 0, 1 = row bands (reduce-scatter)
    // CUDA graph of one Whitted render (all lanes, all batches): a render is ~20 launches per batch and the host
    // needs ~4.5 us per launch, which bounds small renders (1/8 of a frame per GPU) - replaying a captured graph does
    // not.  Keyed by every launch parameter; camera and seed live in a device block so they may change between replays
    int graph = 1;
    int sppm_lanes = 0;           // sub-ranges of each SPPM pass on concurrent streams (0: by scene size)
    int sppm_pipeline = 4;        // SPPM iterations in flight (camera pass / photon tracing of it+1 overlap grid, deposits, collectives of it)
    int deal = -2;                // groups of tiles dealt round-robin to the batches: g > 0 tiles, -r: r tile rows, 0: contiguous bands
    cudaGraphExec_t wh_graph = nullptr;
    std::string wh_graph_key;
    unsigned long long wh_graph_launches[3] = {0, 0, 0};
    std::vector<int> wh_tiles;              // the tile list currently in b_misc[1] (uploaded again only when it changes)
    void* wh_tiles_dev = nullptr;   // kernel / extend / shadow launches one replay stands for

    // scene
    bool have_scene = false;
    DeviceScene scene{};
    DevBuf b_nodes, b_pairs, b_prims, b_tnorm, b_spheres, b_materials, b_lights;
    DevBuf b_shadow;              // the shadow tree's pair records (scene.shadow_pairs), 64 B per primitive
    // trace_scene_upload_mesh_device (upload_device.cu): the LBVH build's scratch, then the pair numbering's and the
    // shadow tree build's (grow-only, so a per-frame rebuild of the same size allocates nothing)
    DevBuf b_build;

    // refit (refit.cu): what trace_scene_refit needs of the last upload.  The host keeps only the BVH-slot -> triangle
    // map; the device topology (parents, pair slots, leaf list) is derived from b_nodes at the first refit after an
    // upload, so scenes that are never refit pay no device memory for it.
    struct Refit {
        std::vector<uint32_t> tri_index;   // [n_prims] trace_prim.index of triangle slots (0 for spheres)
        DevBuf slot_tri_dev;               // the same map already on the device (a device mesh upload), used when
        bool slot_tri_on_device = false;   // slot_tri_on_device: then tri_index is empty
        int64_t n_tris = 0, n_spheres = 0, n_pairs = 0;
        bool topo_ready = false;
        DevBuf topo, stage, sphere_bounds;
        // carved out of `topo` (refit.cu)
        int32_t* parent = nullptr;         // [n_nodes] parent node, -1 at the root
        uint32_t* up = nullptr;            // [n_nodes] 2 * parent's pair index + child slot (0: first, 1: second)
        uint32_t* pair_of = nullptr;       // [n_nodes] interior: its pair index (exclusive scan of "is interior")
        uint32_t* leaves = nullptr;        // [n_nodes - n_pairs] leaf node ids
        uint8_t* empty = nullptr;          // [n_nodes] subtree holds no primitive (per call)
        uint32_t* arrive = nullptr;        // [n_pairs] arrival counters (reset per call)
        uint32_t* slot_tri = nullptr;      // [n_prims] tri_index on the device
        uint32_t* status = nullptr;        // [0] NaN vertex seen
        // the shadow tree's topology, derived from its pair records at the first refit after an upload (refit.cu)
        bool shadow_topo_ready = false;
        DevBuf shadow_topo;
        uint32_t* shadow_up_pair = nullptr;   // [n_prims - 1] 2 * parent pair + slot, ~0 at the root
        uint32_t* shadow_up_prim = nullptr;   // [n_prims] 2 * pair + slot holding the primitive's leaf
        uint32_t* shadow_arrive = nullptr;    // [n_prims - 1] arrival counters (reset per call)
    } refit;

    // scratch
    DevBuf b_query[4];            // ray query staging
    DevBuf b_queue[16];           // wavefront queues
    DevBuf b_misc[8];
    DevBuf b_counters;            // int counters + u64 stats block
    int* h_flags = nullptr;       // pinned host mirror of [overflow, error]

    trace_stats stats{};
    unsigned long long shadow_fallbacks = 0;   // any-hit rays the shadow walk handed to the reference walk (trace_get_shadow_fallbacks)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, evk0 = nullptr, evk1 = nullptr;
    // per-launch CUDA-event timing of the traversal kernels (option "time_kernels"), resolved after a stream sync
    struct KernelEvent { cudaEvent_t a, b; int kind, lane; };
    std::vector<KernelEvent> kev;
    size_t kev_used = 0;
    void kev_begin(int kind) {
        if (!time_kernels) return;
        if (kev_used == kev.size()) { KernelEvent e; cudaEventCreate(&e.a); cudaEventCreate(&e.b); e.kind = kind; kev.push_back(e); }
        kev[kev_used].kind = kind;
        kev[kev_used].lane = cur_lane;
        cudaEventRecord(kev[kev_used].a, cur_stream);
    }
    void kev_end() {
        if (!time_kernels) return;
        cudaEventRecord(kev[kev_used].b, cur_stream);
        kev_used++;
    }
    void kev_collect() {      // call after the stream has been synchronised
        // debugging aid: TRACE_CUDA_TIMELINE=<file> appends "lane kind start_ms end_ms" (relative to the first
        // timed launch) for every timed traversal launch - a poor man's timeline of how the lanes overlap
        const char* tl_path = getenv("TRACE_CUDA_TIMELINE");
        FILE* tl = (tl_path && kev_used) ? fopen(tl_path, "a") : nullptr;
        if (tl) fprintf(tl, "# render\n");
        for (size_t i = 0; i < kev_used; ++i) {
            float ms = 0.0f;
            cudaEventSynchronize(kev[i].b);                 // (launches on side streams may still be running)
            if (tl) {
                float t0 = 0.0f, t1 = 0.0f;
                if (cudaEventElapsedTime(&t0, kev[0].a, kev[i].a) == cudaSuccess && cudaEventElapsedTime(&t1, kev[0].a, kev[i].b) == cudaSuccess)
                    fprintf(tl, "%d %d %.4f %.4f\n", kev[i].lane, kev[i].kind, t0, t1);
            }
            if (cudaEventElapsedTime(&ms, kev[i].a, kev[i].b) == cudaSuccess) {
                const int k = kev[i].kind;
                if (k == TRACE_K_EXTEND) { stats.ms_extend += ms; stats.extend_launches++; }
                else if (k == TRACE_K_SHADOW) { stats.ms_shadow += ms; stats.shadow_launches++; }
                if (k >= 0 && k < TRACE_K_COUNT) { stats.ms_kind[k] += ms; stats.launches_kind[k]++; }
            }
        }
        if (tl) fclose(tl);
        kev_used = 0;
    }

    SppmState* sppm = nullptr;
    std::map<const void*, int> occupancy_cache;   // resident CTAs per SM of each kernel on THIS device

    int fail(const char* fmt, ...) {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof(buf), fmt, ap);
        va_end(ap);
        err = buf;
        return 1;
    }
};

#define TR_CUDA(ctx, call)                                                                  \
    do {                                                                                    \
        cudaError_t e__ = (call);                                                           \
        if (e__ != cudaSuccess) return (ctx)->fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)

// u64 device stats block layout (ctx->b_counters, after the int counters)
enum { ST_RAYS_EXTEND = 0, ST_RAYS_SHADOW = 1, ST_NODES = 2, ST_PRIMS = 3, ST_DEPOSITS = 4, ST_CANDIDATES = 5, ST_REQUESTS = 6, ST_GRID_ITEMS = 7, ST_PRIMARY_RAYS = 8, ST_PRIMARY_HITS = 9, ST_SHADOW_FALLBACKS = 10, ST_COUNT = 12 };
// the traversal kernels get `counters` = stats + ST_NODES; the shadow walk counts its fallbacks at this offset from it
static_assert(ST_SHADOW_FALLBACKS - ST_NODES == 8, "TR_COUNTER_SHADOW_FALLBACKS (traverse.cuh)");
static const int TR_INT_COUNTERS = 128;    // ints at the start of b_counters (64..127: work counters of persistent launches)
// int counter slots: [1 .. TR_MAX_DEPTH] ray-queue length per bounce level, [32] shadow / deposit-request queue
enum { IC_OVERFLOW = 60, IC_ERROR = 61, IC_OVERFLOW_SHADOW = 62, IC_OVERFLOW_DEPOSIT = 63 };
enum { IC_BACK = 33 };     // [IC_BACK + level]: rays pushed from the BACK of bounce level `level`'s queue (Whitted, wavefront.cuh)
// deepest path any entry point accepts (the per-level queue counters live in slots 1..31 of a lane's counter block)
static const int TR_MAX_DEPTH = 24;

// b_counters layout: [lane 0 ints][u64 stats][lane 1 ints][lane 2 ints]...
inline size_t ctx_counter_bytes() {
    return TR_INT_COUNTERS * sizeof(int) * trace_ctx::MAX_LANES + ST_COUNT * sizeof(unsigned long long);
}
inline int* ctx_icounters_lane(trace_ctx* c, int lane) {
    char* base = c->b_counters.as<char>();
    if (lane == 0) return reinterpret_cast<int*>(base);
    return reinterpret_cast<int*>(base + TR_INT_COUNTERS * sizeof(int) + ST_COUNT * sizeof(unsigned long long) +
                                  (size_t)(lane - 1) * TR_INT_COUNTERS * sizeof(int));
}
inline int* ctx_icounters(trace_ctx* c) { return ctx_icounters_lane(c, c->cur_lane); }
inline unsigned long long* ctx_stats64(trace_ctx* c) {
    return reinterpret_cast<unsigned long long*>(c->b_counters.as<char>() + TR_INT_COUNTERS * sizeof(int));
}

// grid for persistent grid-stride kernels: a multiple of the SM count
inline int persistent_grid(const trace_ctx* c, int blocks_per_sm) { return c->num_sms * blocks_per_sm; }

// Grid = SM count x resident CTAs per SM of THIS kernel (occupancy API), so a grid-stride kernel runs as exactly one
// full wave: with a fixed 16 CTAs/SM the 69-register traversal kernels (7 resident) ran 2.29 waves, the last one 29 %
// full (ncu: sm__warps_active 29 % of peak against a 44 % theoretical).
#ifdef __CUDACC__
template <class K>
inline int occupancy_grid(trace_ctx* c, K kernel, int block_size) {
    // cached per context (one context = one device, calls on a context are serialised by the caller)
    const void* key = (const void*)kernel;
    auto it = c->occupancy_cache.find(key);
    int per_sm;
    if (it != c->occupancy_cache.end()) per_sm = it->second;
    else {
        per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block_size, 0) != cudaSuccess || per_sm < 1) per_sm = 4;
        c->occupancy_cache[key] = per_sm;
    }
    return c->num_sms * per_sm;
}
#endif

#include <type_traits>
// Picks the kernel instantiation for the context's (slab, count_nodes, leaf_wait): f(slab, count, wait) gets them as
// integral constants.  Counting is only built for the plain loop (the counts do not depend on the loop shape).
template <class F>
static void trav_dispatch(const trace_ctx* c, F f) {
    using std::integral_constant;
    const int w = c->count_nodes ? 0 : c->leaf_wait;
    if (c->count_nodes) {
        if (c->slab == 0) f(integral_constant<int, 0>{}, integral_constant<bool, true>{}, integral_constant<int, 0>{});
        else if (c->slab == 2) f(integral_constant<int, 2>{}, integral_constant<bool, true>{}, integral_constant<int, 0>{});
        else f(integral_constant<int, 1>{}, integral_constant<bool, true>{}, integral_constant<int, 0>{});
        return;
    }
    if (c->slab == 1) { f(integral_constant<int, 1>{}, integral_constant<bool, false>{}, integral_constant<int, 0>{}); return; }
#define TR_WAIT_CASE(S, W) if (c->slab == S && w == W) { f(integral_constant<int, S>{}, integral_constant<bool, false>{}, integral_constant<int, W>{}); return; }
    TR_WAIT_CASE(2, -1) TR_WAIT_CASE(0, -1)
    TR_WAIT_CASE(2, 8) TR_WAIT_CASE(2, 16) TR_WAIT_CASE(2, 32) TR_WAIT_CASE(2, 4)
    TR_WAIT_CASE(0, 8) TR_WAIT_CASE(0, 16)
#undef TR_WAIT_CASE
    if (c->slab == 0) f(integral_constant<int, 0>{}, integral_constant<bool, false>{}, integral_constant<int, 0>{});
    else f(integral_constant<int, 2>{}, integral_constant<bool, false>{}, integral_constant<int, 0>{});
}

// The scene as an any-hit launch sees it: the shadow tree only with the option on, the guarded test and the pair walk
// (the walk it falls back to, and the guard its admission test relies on)
inline DeviceScene shadow_launch_scene(const trace_ctx* c, DeviceScene sc) {
    if (!(c->shadow_tree && c->slab == 2 && c->leaf_wait == -1 /* TR_WALK_PAIR */)) sc.shadow_pairs = nullptr;
    return sc;
}

// implemented in api.cu
int ctx_device_film(trace_ctx* ctx, const trace_film_desc* film, DeviceFilm* out, DevBuf* table_buf);
void ctx_device_camera(const trace_camera* cam, DeviceCamera* out);
int ctx_pull_stats(trace_ctx* ctx);
// implemented in comm.cpp: float32 collectives of the context's communicator, enqueued on ctx->stream
int comm_reduce_sum(trace_ctx* ctx, const float* send, float* recv, size_t count, int root);
int comm_reduce_scatter_sum(trace_ctx* ctx, const float* send, float* recv, size_t recv_count);
int comm_allreduce_sum(trace_ctx* ctx, float* buf, size_t count);
int comm_allreduce_sum_int(trace_ctx* ctx, int* buf, size_t count);
int comm_allgather(trace_ctx* ctx, const float* send, float* recv, size_t send_count);
int comm_reduce_sum_via_scatter(trace_ctx* ctx, float* buf, size_t chunk, int root);
int comm_p2p_exchange(trace_ctx* ctx, void* base, std::vector<void*>& peers_out, std::vector<void*>& opened_out, int* all_ok);
void comm_p2p_close(trace_ctx* ctx);
int comm_group_begin(trace_ctx* ctx);
int comm_group_end(trace_ctx* ctx);
// implemented in whitted.cu / sppm.cu
int whitted_render_device(trace_ctx* ctx, const trace_camera* cam, const trace_film_desc* film, int spp, int max_depth,
                          uint64_t seed, float* film_xyzw_device);
void sppm_free(trace_ctx* ctx);
void sppm_end_session(trace_ctx* ctx);
void whitted_film_range(const trace_ctx* ctx, long long npix, long long* p0, long long* p1);
// implemented in bvh_gpu.cu: the shadow tree over uploaded primitive records (0, 5 NaN, 6 too deep, 7 CUDA error), in
// `scratch` (lbvh_scratch_bytes(n) bytes) or, with nullptr, an allocation of its own; the device mesh build's steps
int shadow_tree_build(cudaStream_t s, const void* prims, int64_t n, void* pairs, void* scratch);
size_t lbvh_scratch_bytes(int64_t n, cudaStream_t s);
int lbvh_mesh_validate(cudaStream_t s, const float* nrm, const uint32_t* mat, int64_t n_materials, int64_t n, void* scratch);
int lbvh_mesh_bounds(cudaStream_t s, const float* v, int64_t n, void* scratch);
int lbvh_mesh_build(cudaStream_t s, int64_t n, int m, void* scratch, int64_t* n_nodes, const uint32_t** order);
int lbvh_mesh_emit(cudaStream_t s, int64_t n, int m, void* scratch, void* nodes);
// implemented in api.cu: the parts of a scene upload that do not depend on where the tree was built
int ctx_pack_materials(trace_ctx* ctx, int64_t n, const trace_material* in, std::vector<DeviceMaterial>& out);
int ctx_pack_lights(trace_ctx* ctx, int64_t n, const trace_light* in, std::vector<DeviceLight>& out);
int ctx_put(trace_ctx* ctx, DevBuf& b, const void* src, size_t bytes);
int ctx_commit_scene(trace_ctx* ctx, int64_t n_nodes, int64_t n_prims, int64_t n_spheres, int64_t n_materials,
                     int64_t n_lights, int64_t n_tris, int64_t n_pairs, uint32_t root_ref, const float* root_box,
                     void* shadow_scratch);
// implemented in refit.cu: waits for every stream of the context (caller's, lanes, SPPM chain / collectives, copies)
int ctx_drain(trace_ctx* ctx);
// implemented in refit.cu: the upload's preorder pair numbering of a device node array (2 float4 per node), pair_of[i] =
// interior nodes before node i, as an exclusive scan of "is interior" (`flag`: n words of scratch; `tmp`:
// pair_scan_bytes(n) bytes of scan scratch)
size_t pair_scan_bytes(int64_t n, cudaStream_t s);
cudaError_t pair_numbering(cudaStream_t s, const float4* nodes, int64_t n, uint32_t* flag, uint32_t* pair_of, void* tmp,
                           size_t tmp_bytes);

// TRACE_BVH_PROFILE=1: CUDA events between the phases of an upload / refit call, printed as one stderr line
struct PhaseTimer {
    bool on = false;
    cudaEvent_t ev[12] = {};
    const char* name[12] = {};
    int n = 0;
    void mark(cudaStream_t s, const char* what) {      // `what` names the phase that ends here
        if (!on || n >= 12) return;
        if (!ev[n]) cudaEventCreate(&ev[n]);
        name[n] = what;
        cudaEventRecord(ev[n++], s);
    }
    void print(const char* head, double wall_ms) {     // after the last mark's work is done
        fprintf(stderr, "%s, wall %.3f ms;", head, wall_ms);
        for (int i = 1; i < n; ++i) {
            float ms = 0.0f;
            cudaEventElapsedTime(&ms, ev[i - 1], ev[i]);
            fprintf(stderr, " %s %.3f ms%s", name[i], ms, i + 1 < n ? "," : "\n");
        }
    }
    ~PhaseTimer() { for (auto e : ev) if (e) cudaEventDestroy(e); }
};
