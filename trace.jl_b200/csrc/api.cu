// api.cu — context, scene upload and the batch ray-query entry points of libtrace_cuda.so (include/trace_cuda.h).
#include <cmath>
#include <cstring>

#include "context.hpp"
#include "shading.cuh"

// ------------------------------------------------------------------ kernels: batch closest-hit / any-hit queries
// One thread per ray, persistent grid-stride loop (grid = multiple of the SM count).  Rays come as two float4 arrays
// {o.xyz, t_max} and {d.xyz, -}; the closest-hit result is one float4 {t, original+1 (bits), b0, b1}.
template <int SLAB, bool COUNT, int WAIT, bool TREE>       // TREE: walk the shadow tree (traverse_closest)
__global__ void __launch_bounds__(128, 8) k_intersect(DeviceScene sc, const float4* __restrict__ ro, const float4* __restrict__ rd,
                                                   long long n, float4* __restrict__ hits, unsigned long long* counters,
                                                   int* error_flag) {
    const int lane = threadIdx.x & 31;
    for (long long base = blockIdx.x * (long long)blockDim.x + (threadIdx.x - lane); base < n; base += (long long)gridDim.x * blockDim.x) {
        const long long i = base + lane;
        const bool valid = i < n;
        const float4 o = valid ? ro[i] : make_float4(0.0f, 0.0f, 0.0f, 0.0f), d = valid ? rd[i] : make_float4(1.0f, 1.0f, 1.0f, 0.0f);
        HitRecord h;
        traverse_closest<SLAB, COUNT, WAIT, TREE>(sc, valid, xyz(o), xyz(d), o.w, h, counters, error_flag);
        if (!valid) continue;
        uint32_t orig = 0;
        if (h.prim) orig = __float_as_uint(__ldg(&sc.prims[3 * (h.prim - 1) + 2]).w) + 1u;
        hits[i] = make_float4(h.prim ? h.t : o.w, __uint_as_float(orig), h.b0, h.b1);
    }
}
template <int SLAB, bool COUNT, int WAIT, bool TREE>       // TREE: walk the shadow tree (wavefront.cuh k_wh_shadow)
__global__ void __launch_bounds__(128, 8) k_occluded(DeviceScene sc, const float4* __restrict__ ro, const float4* __restrict__ rd,
                                                  long long n, uint8_t* __restrict__ out, unsigned long long* counters,
                                                  int* error_flag) {
    const int lane = threadIdx.x & 31;
    for (long long base = blockIdx.x * (long long)blockDim.x + (threadIdx.x - lane); base < n; base += (long long)gridDim.x * blockDim.x) {
        const long long i = base + lane;
        const bool valid = i < n;
        const float4 o = valid ? ro[i] : make_float4(0.0f, 0.0f, 0.0f, 0.0f), d = valid ? rd[i] : make_float4(1.0f, 1.0f, 1.0f, 0.0f);
        bool occ;
        if (TREE) occ = valid && traverse_shadow<COUNT>(sc, xyz(o), xyz(d), o.w, counters, error_flag);
        else {
            HitRecord h;
            occ = traverse_any<SLAB, true, COUNT, WAIT>(sc, valid, xyz(o), xyz(d), o.w, h, counters, error_flag);
        }
        if (valid) out[i] = occ ? 1 : 0;
    }
}

// ------------------------------------------------------------------ context
extern "C" int trace_abi_version(void) { return TRACE_ABI_VERSION; }

extern "C" int trace_create(trace_ctx** out, int device, void* cuda_stream) {
    if (!out) return 1;
    *out = nullptr;
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || device < 0 || device >= n_dev) return 2;   // no CPU fallback
    if (cudaSetDevice(device) != cudaSuccess) return 3;
    trace_ctx* c = new trace_ctx();
    c->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) c->num_sms = prop.multiProcessorCount;
    if (cuda_stream) { c->stream = (cudaStream_t)cuda_stream; c->own_stream = false; }
    else {
        if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return 4; }
        c->own_stream = true;
    }
    bool ok = cudaEventCreate(&c->ev0) == cudaSuccess && cudaEventCreate(&c->ev1) == cudaSuccess &&
              cudaEventCreate(&c->evk0) == cudaSuccess && cudaEventCreate(&c->evk1) == cudaSuccess;
    ok = ok && c->b_counters.ensure(ctx_counter_bytes()) == cudaSuccess;
    c->cur_stream = c->stream;
    ok = ok && cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&c->ev_copy, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking) == cudaSuccess;
    {
        int least = 0, greatest = 0;
        cudaDeviceGetStreamPriorityRange(&least, &greatest);
        ok = ok && cudaStreamCreateWithPriority(&c->chain_stream, cudaStreamNonBlocking, greatest) == cudaSuccess;
        ok = ok && cudaStreamCreateWithPriority(&c->coll_stream, cudaStreamNonBlocking, greatest) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&c->ev_chain, cudaEventDisableTiming) == cudaSuccess;
    }
    for (int l = 0; l < trace_ctx::MAX_LANES && ok; ++l)
        ok = cudaStreamCreateWithFlags(&c->side[l], cudaStreamNonBlocking) == cudaSuccess &&
             cudaEventCreateWithFlags(&c->ev_join[l], cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaMallocHost((void**)&c->h_flags, 64 * sizeof(int)) == cudaSuccess;
    if (ok) ok = cudaMemsetAsync(c->b_counters.p, 0, c->b_counters.bytes, c->stream) == cudaSuccess;
    if (!ok) { trace_destroy(c); return 5; }
    memset(&c->stats, 0, sizeof(c->stats));
    *out = c;
    return 0;
}

extern "C" void trace_destroy(trace_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    sppm_free(c);
    trace_comm_destroy(c);
    DevBuf* all[] = {&c->b_nodes, &c->b_pairs, &c->b_prims, &c->b_tnorm, &c->b_spheres, &c->b_materials, &c->b_lights, &c->b_counters,
                     &c->b_shadow, &c->refit.topo, &c->refit.stage, &c->refit.sphere_bounds, &c->refit.shadow_topo,
                     &c->refit.slot_tri_dev, &c->b_build};
    for (DevBuf* b : all) b->release();
    for (auto& b : c->b_query) b.release();
    for (auto& b : c->b_queue) b.release();
    c->p2p_film.release();
    for (auto& b : c->b_misc) b.release();
    for (auto& e : c->kev) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); }
    for (int l = 0; l < trace_ctx::MAX_LANES; ++l) { if (c->side[l]) cudaStreamDestroy(c->side[l]); if (c->ev_join[l]) cudaEventDestroy(c->ev_join[l]); }
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_copy) cudaEventDestroy(c->ev_copy);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->chain_stream) cudaStreamDestroy(c->chain_stream);
    if (c->coll_stream) cudaStreamDestroy(c->coll_stream);
    if (c->ev_chain) cudaEventDestroy(c->ev_chain);
    if (c->wh_graph) cudaGraphExecDestroy(c->wh_graph);
    if (c->h_flags) cudaFreeHost(c->h_flags);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->evk0) cudaEventDestroy(c->evk0);
    if (c->evk1) cudaEventDestroy(c->evk1);
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

extern "C" const char* trace_last_error(const trace_ctx* c) { return c ? c->err.c_str() : "null context"; }

extern "C" int trace_set_option(trace_ctx* c, const char* key, int64_t v) {
    if (!c || !key) return 1;
    if (!strcmp(key, "slab")) { if (v < 0 || v > 2) return c->fail("slab must be 0 (literal), 1 (textbook) or 2 (guarded)"); c->slab = (int)v; }
    else if (!strcmp(key, "batch")) { if (v < 1024) return c->fail("batch too small"); c->batch = v; }
    else if (!strcmp(key, "count_nodes")) { if (v < 0 || v > 2) return c->fail("count_nodes must be 0, 1 (closest hits on the reference tree) or 2 (the walks the default path runs)"); c->count_nodes = (int)v; }
    else if (!strcmp(key, "persist")) { if (v != 0) return c->fail("persist: the dynamic-ray-fetch kernels were measured slower in both rounds and removed (profiles/r2_experiments.md)"); }
    else if (!strcmp(key, "film_mode")) { if (v != 0 && v != 1) return c->fail("film_mode must be 0 (whole film on rank 0) or 1 (one band per rank)"); c->film_mode = (int)v; }
    else if (!strcmp(key, "film_p2p")) { c->film_p2p = v != 0; }
    else if (!strcmp(key, "film_sum")) { if (v < 0 || v > 2) return c->fail("film_sum must be 0 (ncclReduce), 1 (ncclAllReduce) or 2 (reduce-scatter + gather)"); c->film_sum = (int)v; }
    else if (!strcmp(key, "sppm_path")) { if (v < 0 || v > TR_MAX_DEPTH) return c->fail("sppm_path must be in [0, %d]", TR_MAX_DEPTH); c->sppm_path = (int)v; }
    else if (!strcmp(key, "fuse_primary")) c->fuse_primary = v != 0;
    else if (!strcmp(key, "walk")) { if (v != 0 && v != 1) return c->fail("walk must be 0 (one node per step, the reference loop) or 1 (pair nodes)"); c->leaf_wait = v ? TR_WALK_PAIR : 0; }
    else if (!strcmp(key, "leaf_wait")) { if (v != 0 && v != 4 && v != 8 && v != 16 && v != 32) return c->fail("leaf_wait must be 0, 4, 8, 16 or 32"); c->leaf_wait = (int)v; }
    else if (!strcmp(key, "lanes")) { if (v < 1 || v > trace_ctx::MAX_LANES) return c->fail("lanes must be in [1, 16]"); c->lanes = (int)v; }
    else if (!strcmp(key, "cap_percent")) { if (v < 100 || v > 1600) return c->fail("cap_percent must be in [100, 1600]"); c->cap_percent = (int)v; }
    else if (!strcmp(key, "time_kernels")) c->time_kernels = v != 0;
    else if (!strcmp(key, "shadow_tree")) c->shadow_tree = v != 0;
    else if (!strcmp(key, "hit_tree")) c->hit_tree = v != 0;
    else if (!strcmp(key, "graph")) c->graph = v != 0;
    else if (!strcmp(key, "sppm_lanes")) { if (v < 0 || v > trace_ctx::MAX_LANES / 2) return c->fail("sppm_lanes must be in [0, 8]"); c->sppm_lanes = (int)v; }
    else if (!strcmp(key, "sppm_chain_priority")) c->sppm_chain_priority = v != 0;
    else if (!strcmp(key, "sppm_pipeline")) { if (v < 1 || v > 8) return c->fail("sppm_pipeline must be in [1, 8]"); c->sppm_pipeline = (int)v; }
    else if (!strcmp(key, "deal")) c->deal = (int)v;
    else if (!strcmp(key, "rank")) { if (c->comm) return c->fail("rank is fixed by trace_comm_init"); c->rank = (int)v; }
    else if (!strcmp(key, "world")) { if (c->comm) return c->fail("world is fixed by trace_comm_init"); if (v < 1) return c->fail("world must be >= 1"); c->world = (int)v; }
    else return c->fail("unknown option '%s'", key);
    if (c->rank < 0 || c->rank >= c->world) { /* validated at render time */ }
    return 0;
}

int ctx_pull_stats(trace_ctx* c) {
    unsigned long long h[ST_COUNT];
    TR_CUDA(c, cudaMemcpyAsync(h, ctx_stats64(c), sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(c, cudaStreamSynchronize(c->stream));
    c->stats.rays_extend = h[ST_RAYS_EXTEND];
    c->stats.rays_shadow = h[ST_RAYS_SHADOW];
    c->stats.nodes_visited = h[ST_NODES];
    c->stats.prims_tested = h[ST_PRIMS];
    c->stats.sppm_deposits = h[ST_DEPOSITS];
    c->stats.sppm_candidates = h[ST_CANDIDATES];
    c->stats.sppm_requests = h[ST_REQUESTS];
    c->stats.sppm_grid_items = h[ST_GRID_ITEMS];
    c->stats.primary_rays = h[ST_PRIMARY_RAYS];
    c->stats.primary_hits = h[ST_PRIMARY_HITS];
    c->shadow_fallbacks = h[ST_SHADOW_FALLBACKS];
    c->hit_fallbacks = h[ST_HIT_FALLBACKS];
    return 0;
}

extern "C" int trace_get_stats(trace_ctx* c, trace_stats* out) {
    if (!c || !out) return 1;
    cudaSetDevice(c->device);
    if (ctx_pull_stats(c)) return 1;
    *out = c->stats;
    return 0;
}
extern "C" int trace_reset_stats(trace_ctx* c) {
    if (!c) return 1;
    cudaSetDevice(c->device);
    TR_CUDA(c, cudaMemsetAsync(c->b_counters.p, 0, c->b_counters.bytes, c->stream));
    memset(&c->stats, 0, sizeof(c->stats));
    return 0;
}
extern "C" int trace_synchronize(trace_ctx* c) {
    if (!c) return 1;
    cudaSetDevice(c->device);
    TR_CUDA(c, cudaStreamSynchronize(c->stream));
    return 0;
}

// ------------------------------------------------------------------ scene upload
static float remap_alpha(float roughness) {         // roughness_to_α, reflection/microfacet.jl:79-84
    roughness = fmaxf(1e-3f, roughness);
    float x = logf(roughness);
    double xd = (double)x;
    float x4 = (float)((xd * xd) * (xd * xd));
    return 1.62142f + 0.819955f * x + 0.1734f * (x * x) + 0.0171201f * (x * x * x) + 0.000640711f * x4;
}

extern "C" int trace_scene_upload(trace_ctx* c, const trace_scene_desc* d) {
    if (!c || !d) return 1;
    cudaSetDevice(c->device);
    if (d->n_nodes < 0 || d->n_prims < 0 || (d->n_nodes > 0 && !d->nodes) || (d->n_prims > 0 && !d->prims))
        return c->fail("scene: bad node / primitive arrays");
    if (d->n_prims >= (1ll << 30)) return c->fail("scene: too many primitives");
    // --- validate + pack on the host
    std::vector<float4> nodes((size_t)d->n_nodes * 2);
    int64_t n_pairs = 0;                                   // pair records (traverse.cuh): one per interior node
    for (int64_t i = 0; i < d->n_nodes; ++i) {
        const trace_bvh_node& n = d->nodes[i];
        if (tr_node_leaf(n.meta)) { if ((int64_t)n.offset + (int64_t)(n.meta & ~TRACE_NODE_LEAF) > d->n_prims) return c->fail("scene: leaf %lld out of range", (long long)i); }
        else if ((int64_t)n.offset >= d->n_nodes || i + 1 >= d->n_nodes) return c->fail("scene: interior node %lld out of range", (long long)i);
        else ++n_pairs;
        float4 a, b;
        a.x = n.bmin[0]; a.y = n.bmin[1]; a.z = n.bmin[2]; a.w = n.bmax[0];
        b.x = n.bmax[1]; b.y = n.bmax[2];
        memcpy(&b.z, &n.offset, 4); memcpy(&b.w, &n.meta, 4);
        nodes[2 * i] = a; nodes[2 * i + 1] = b;
    }
    // device-only meta bit 29: "an analytic sphere lives in this subtree" (see traverse.cuh). Preorder => children have
    // larger indices than their parent, so one reverse sweep propagates it.
    {
        std::vector<uint8_t> below((size_t)d->n_nodes, 0);
        for (int64_t i = d->n_nodes - 1; i >= 0; --i) {
            const trace_bvh_node& n = d->nodes[i];
            uint8_t f = 0;
            if (tr_node_leaf(n.meta)) {
                const uint32_t cnt = n.meta & ~TRACE_NODE_LEAF;
                if (cnt > TR_NODE_COUNT_MASK) return c->fail("scene: leaf %lld holds too many primitives", (long long)i);
                for (uint32_t k = 0; k < cnt; ++k) if (d->prims[n.offset + k].kind == TRACE_PRIM_SPHERE) f = 1;
            } else f = below[i + 1] | below[n.offset];
            below[i] = f;
            if (f) { uint32_t m; memcpy(&m, &nodes[2 * i + 1].w, 4); m |= TR_NODE_SPHERE_BELOW; memcpy(&nodes[2 * i + 1].w, &m, 4); }
        }
    }
    std::vector<float4> prims((size_t)d->n_prims * 3), tnorm((size_t)d->n_prims * 3);
    std::vector<uint32_t> tri_index((size_t)d->n_prims, 0u);        // kept for trace_scene_refit
    for (int64_t i = 0; i < d->n_prims; ++i) {
        const trace_prim& p = d->prims[i];
        float4 A = make_float4(0, 0, 0, 0), B = A, C = A, N0 = A, N1 = A, N2 = A;
        uint32_t tag = 0, flags = 0;
        if (p.kind == TRACE_PRIM_TRIANGLE) {
            if ((int64_t)p.index >= d->n_tris || !d->tri_vertices) return c->fail("scene: triangle index out of range");
            const float* v = d->tri_vertices + 9 * (size_t)p.index;
            A.x = v[0]; A.y = v[1]; A.z = v[2]; B.x = v[3]; B.y = v[4]; B.z = v[5]; C.x = v[6]; C.y = v[7]; C.z = v[8];
            if (tri_degenerate(f3(v[0], v[1], v[2]), f3(v[3], v[4], v[5]), f3(v[6], v[7], v[8]))) tag = TR_PRIM_DEGENERATE_BIT;
            tri_index[i] = p.index;
            flags = d->tri_flags ? d->tri_flags[p.index] : 0;
            if (!d->tri_normals) flags &= ~(uint32_t)TRACE_TRI_HAS_NORMALS;
            if (flags & TRACE_TRI_HAS_NORMALS) {
                const float* nn = d->tri_normals + 9 * (size_t)p.index;
                N0.x = nn[0]; N0.y = nn[1]; N0.z = nn[2]; N1.x = nn[3]; N1.y = nn[4]; N1.z = nn[5]; N2.x = nn[6]; N2.y = nn[7]; N2.z = nn[8];
            }
        } else if (p.kind == TRACE_PRIM_SPHERE) {
            if ((int64_t)p.index >= d->n_spheres) return c->fail("scene: sphere index out of range");
            tag = TR_PRIM_SPHERE_BIT | p.index;
        } else return c->fail("scene: unknown primitive kind %u", p.kind);
        if (p.material != 0xFFFFFFFFu && (int64_t)p.material >= d->n_materials) return c->fail("scene: material index out of range");
        memcpy(&A.w, &tag, 4); memcpy(&B.w, &p.material, 4); memcpy(&C.w, &p.original, 4);
        memcpy(&N0.w, &flags, 4);
        prims[3 * i] = A; prims[3 * i + 1] = B; prims[3 * i + 2] = C;
        tnorm[3 * i] = N0; tnorm[3 * i + 1] = N1; tnorm[3 * i + 2] = N2;
    }
    if (n_pairs > TR_REF_INDEX_MASK) return c->fail("scene: too many interior nodes");
    std::vector<DeviceSphere> spheres((size_t)d->n_spheres);
    for (int64_t i = 0; i < d->n_spheres; ++i) {
        static_assert(sizeof(DeviceSphere) == sizeof(trace_sphere), "sphere layout");
        memcpy(&spheres[i], &d->spheres[i], sizeof(trace_sphere));
    }
    std::vector<DeviceMaterial> mats;
    std::vector<DeviceLight> lights;
    if (ctx_pack_materials(c, d->n_materials, d->materials, mats) || ctx_pack_lights(c, d->n_lights, d->lights, lights)) return 1;
    const size_t scan_bytes = d->n_nodes > 0 ? pair_scan_bytes(d->n_nodes, c->stream) : 1;
    if (!scan_bytes) return c->fail("scene: cannot size the pair scan");
    // --- upload; then the pair records and last-of-leaf bits, on the device (upload_device.cu)
    TR_CUDA(c, cudaStreamSynchronize(c->stream));
    if (ctx_put(c, c->b_nodes, nodes.data(), nodes.size() * sizeof(float4)) ||
        ctx_put(c, c->b_prims, prims.data(), prims.size() * sizeof(float4)) ||
        ctx_put(c, c->b_tnorm, tnorm.data(), tnorm.size() * sizeof(float4)) ||
        ctx_put(c, c->b_spheres, spheres.data(), spheres.size() * sizeof(DeviceSphere)) ||
        ctx_put(c, c->b_materials, mats.data(), mats.size() * sizeof(DeviceMaterial)) ||
        ctx_put(c, c->b_lights, lights.data(), lights.size() * sizeof(DeviceLight)))
        return 1;
    TR_CUDA(c, c->b_pairs.ensure(n_pairs ? (size_t)n_pairs * 4 * sizeof(float4) : 16));
    if (d->n_nodes > 0) {
        TR_CUDA(c, c->b_build.ensure(pair_scratch_bytes(d->n_nodes, scan_bytes)));
        if (ctx_pack_pairs(c, d->n_nodes, c->b_build.as<char>(), scan_bytes)) return 1;
    }
    TR_CUDA(c, cudaStreamSynchronize(c->stream));      // host staging vectors die at return
    c->refit.tri_index.swap(tri_index);
    c->refit.slot_tri_on_device = false;
    return ctx_commit_scene(c, d->n_nodes, d->n_prims, d->n_spheres, mats, lights, d->n_tris, n_pairs, nodes.data(), nullptr);
}

int ctx_pack_materials(trace_ctx* c, int64_t n, const trace_material* in, std::vector<DeviceMaterial>& out) {
    if (n < 0 || (n > 0 && !in)) return c->fail("scene: bad material array");
    out.resize((size_t)n);
    for (int64_t i = 0; i < n; ++i) {
        const trace_material& m = in[i];
        DeviceMaterial dm;
        memset(&dm, 0, sizeof(dm));
        dm.kind = m.kind;
        for (int k = 0; k < 3; ++k) { dm.a[k] = m.a[k]; dm.b[k] = m.b[k]; }
        dm.eta = m.eta;
        if (m.kind == TRACE_MAT_MATTE) {
            // sigma = clamp(sigma, 0, 90); sigma == 0 -> Lambertian, else Oren-Nayar with A, B (microfacet.jl:12-18)
            const float sigma = m.rough_u > 90.0f ? 90.0f : (m.rough_u < 0.0f ? 0.0f : m.rough_u);
            dm.specular = sigma == 0.0f ? 1u : 0u;
            const float sr = sigma * (3.1415927f / 180.0f), s2 = sr * sr;
            dm.alpha_u = 1.0f - (s2 / (2.0f * (s2 + 0.33f)));
            dm.alpha_v = 0.45f * s2 / (s2 + 0.09f);
        } else if (m.kind == TRACE_MAT_GLASS) {
            dm.specular = (m.rough_u == 0.0f && m.rough_v == 0.0f) ? 1u : 0u;
            const float ru = m.remap ? remap_alpha(m.rough_u) : m.rough_u, rv = m.remap ? remap_alpha(m.rough_v) : m.rough_v;
            dm.alpha_u = fmaxf(1e-3f, ru); dm.alpha_v = fmaxf(1e-3f, rv);      // material.jl:93-98, microfacet.jl:58-62
        } else if (m.kind == TRACE_MAT_PLASTIC) {
            float r = m.remap ? remap_alpha(m.rough_u) : m.rough_u;
            dm.alpha_u = dm.alpha_v = fmaxf(1e-3f, r);           // TrowbridgeReitzDistribution clamps, microfacet.jl:58-62
        } else if (m.kind != TRACE_MAT_MIRROR) return c->fail("material %lld: unknown kind %u", (long long)i, m.kind);
        out[i] = dm;
    }
    return 0;
}

int ctx_pack_lights(trace_ctx* c, int64_t n, const trace_light* in, std::vector<DeviceLight>& out) {
    if (n < 0 || (n > 0 && !in)) return c->fail("scene: bad light array");
    out.resize((size_t)n);
    for (int64_t i = 0; i < n; ++i) {
        const trace_light& l = in[i];
        DeviceLight dl;
        dl.kind = l.kind;
        memcpy(dl.m, l.m, sizeof(dl.m)); memcpy(dl.inv_m, l.inv_m, sizeof(dl.inv_m));
        for (int k = 0; k < 3; ++k) { dl.I[k] = l.I[k]; dl.pos[k] = l.position[k]; }
        dl.cos_total = l.cos_total_width; dl.cos_falloff = l.cos_falloff_start;
        if (l.kind != TRACE_LIGHT_POINT && l.kind != TRACE_LIGHT_SPOT && l.kind != TRACE_LIGHT_DIRECTIONAL)
            return c->fail("light %lld: unknown kind", (long long)i);
        out[i] = dl;
    }
    return 0;
}

// host -> device into a grow-only scene buffer (16 bytes for an empty array), on the context's stream
int ctx_put(trace_ctx* c, DevBuf& b, const void* src, size_t bytes) {
    TR_CUDA(c, b.ensure(bytes ? bytes : 16));
    if (bytes) TR_CUDA(c, cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, c->stream));
    return 0;
}

// The walks' root reference (DeviceScene::root_ref) from the root node record: pair 0, or a single leaf by its first
// primitive (a zero-primitive leaf by 0: it is never entered)
static uint32_t root_ref_of(const float4* root) {
    uint32_t offset, meta;
    memcpy(&offset, &root[1].z, 4); memcpy(&meta, &root[1].w, 4);
    if (!tr_node_leaf(meta)) return 0u;
    return TR_REF_LEAF | (tr_node_count(meta) ? offset : 0u);
}

// The tail of every upload, once the scene buffers hold the new scene: the shadow tree, the scene as the base of
// later attaches (trace_scene_attach_mesh_device, upload_device.cu; `mats` and `lights` are taken), then
// ctx_publish_scene.  The caller sets the refit's slot -> triangle map.
int ctx_commit_scene(trace_ctx* c, int64_t n_nodes, int64_t n_prims, int64_t n_spheres, std::vector<DeviceMaterial>& mats,
                     std::vector<DeviceLight>& lights, int64_t n_tris, int64_t n_pairs, const float4* root,
                     void* shadow_scratch) {
    // the shadow tree (traverse.cuh, traverse_shadow): built on the device from the uploaded primitive records.  Scenes
    // with analytic spheres have none (the guard its walk admits nodes with is off below spheres); neither has a scene
    // uploaded with option shadow_tree 0
    int depth = 0;
    bool shadow = false;
    if (c->shadow_tree && n_spheres == 0 && n_prims >= 2) {
        TR_CUDA(c, c->b_shadow.ensure((size_t)(n_prims - 1) * 4 * sizeof(float4)));
        const int rc = shadow_tree_build(c->stream, c->b_prims.p, n_prims, c->b_shadow.p, shadow_scratch, &depth);
        if (rc == 0) shadow = true;
        else if (rc != LBVH_NAN_BOUND && rc != LBVH_TOO_DEEP) return c->fail("scene: shadow tree build failed (CUDA error)");
    }
    auto& B = c->base;
    B.n_nodes = n_nodes; B.n_pairs = n_pairs; B.n_prims = n_prims; B.n_tris = n_tris; B.n_spheres = n_spheres;
    B.shadow_depth = shadow ? depth : (n_prims == 1 ? 1 : 0);
    B.moved = false;
    c->slots.clear();
    B.materials.swap(mats);
    B.lights.swap(lights);
    ctx_publish_scene(c, n_nodes, n_prims, n_spheres, (int64_t)B.materials.size(), (int64_t)B.lights.size(), n_tris, n_pairs,
                      root, shadow);
    return 0;
}

// The DeviceScene over the scene buffers, root_ref and scene_scale from the root node record, the shadow tree in
// b_shadow when `shadow`, the refit state and the end of any SPPM session
void ctx_publish_scene(trace_ctx* c, int64_t n_nodes, int64_t n_prims, int64_t n_spheres, int64_t n_materials,
                       int64_t n_lights, int64_t n_tris, int64_t n_pairs, const float4* root, bool shadow) {
    DeviceScene& s = c->scene;
    s.nodes = c->b_nodes.as<float4>(); s.pairs = c->b_pairs.as<float4>(); s.prims = c->b_prims.as<float4>(); s.tnorm = c->b_tnorm.as<float4>();
    s.spheres = c->b_spheres.as<DeviceSphere>(); s.materials = c->b_materials.as<DeviceMaterial>();
    s.lights = c->b_lights.as<DeviceLight>();
    s.n_nodes = (int)n_nodes; s.n_prims = (int)n_prims; s.n_spheres = (int)n_spheres;
    s.n_materials = (int)n_materials; s.n_lights = (int)n_lights;
    s.root_ref = n_nodes > 0 ? root_ref_of(root) : 0u;
    s.scene_scale = 0.0f;
    if (n_nodes > 0) {
        const float root_box[6] = {root[0].x, root[0].y, root[0].z, root[0].w, root[1].x, root[1].y};   // min xyz, max xyz
        for (int k = 0; k < 6; ++k) {
            const float a = fabsf(root_box[k]);
            if (std::isfinite(a)) s.scene_scale = fmaxf(s.scene_scale, a);
        }
    }
    s.shadow_pairs = shadow ? c->b_shadow.as<float4>() : nullptr;
    c->have_scene = true;
    c->refit.n_tris = n_tris; c->refit.n_spheres = n_spheres; c->refit.n_pairs = n_pairs;
    c->refit.topo_ready = false;
    c->refit.shadow_topo_ready = false;
    sppm_end_session(c);
}

int ctx_drain(trace_ctx* c) {
    TR_CUDA(c, cudaStreamSynchronize(c->stream));
    for (int l = 0; l < trace_ctx::MAX_LANES; ++l) if (c->side[l]) TR_CUDA(c, cudaStreamSynchronize(c->side[l]));
    cudaStream_t more[] = {c->chain_stream, c->coll_stream, c->copy_stream};
    for (cudaStream_t s : more) if (s) TR_CUDA(c, cudaStreamSynchronize(s));
    return 0;
}

extern "C" int trace_scene_shadow_tree(trace_ctx* c, int64_t* n_pairs, void* pairs_out) {
    if (!c || !n_pairs) return 1;
    cudaSetDevice(c->device);
    if (!c->have_scene) return c->fail("no scene uploaded");
    *n_pairs = c->scene.shadow_pairs ? c->scene.n_prims - 1 : 0;
    if (pairs_out && *n_pairs) {
        TR_CUDA(c, cudaMemcpyAsync(pairs_out, c->scene.shadow_pairs, (size_t)*n_pairs * 4 * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
        TR_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    return 0;
}

extern "C" int trace_get_shadow_fallbacks(trace_ctx* c, uint64_t* out) {
    if (!c || !out) return 1;
    cudaSetDevice(c->device);
    if (ctx_pull_stats(c)) return 1;
    *out = c->shadow_fallbacks;
    return 0;
}

extern "C" int trace_get_hit_fallbacks(trace_ctx* c, uint64_t* out) {
    if (!c || !out) return 1;
    cudaSetDevice(c->device);
    if (ctx_pull_stats(c)) return 1;
    *out = c->hit_fallbacks;
    return 0;
}

// ------------------------------------------------------------------ film / camera helpers shared with the integrators
void ctx_device_camera(const trace_camera* cam, DeviceCamera* out) {
    memcpy(out->r2c, cam->raster_to_camera, sizeof(out->r2c));
    memcpy(out->c2w, cam->camera_to_world, sizeof(out->c2w));
    out->lens_radius = cam->lens_radius; out->focal_distance = cam->focal_distance;
    out->shutter_open = cam->shutter_open; out->shutter_close = cam->shutter_close;
}

int ctx_device_film(trace_ctx* c, const trace_film_desc* f, DeviceFilm* o, DevBuf* table_buf) {
    if (f->crop_x1 < f->crop_x0 || f->crop_y1 < f->crop_y0) return c->fail("film: empty crop window");
    if (!(f->filter_radius[0] > 0.0f) || !(f->filter_radius[1] > 0.0f)) return c->fail("film: bad filter radius");
    o->crop_x0 = f->crop_x0; o->crop_y0 = f->crop_y0; o->crop_x1 = f->crop_x1; o->crop_y1 = f->crop_y1;
    o->rx = f->filter_radius[0]; o->ry = f->filter_radius[1];
    o->inv_rx = 1.0f / o->rx; o->inv_ry = 1.0f / o->ry;
    // get_sample_bounds, film.jl:68-73
    o->sb_x0 = (int)floorf((float)f->crop_x0 + 0.5f - o->rx); o->sb_y0 = (int)floorf((float)f->crop_y0 + 0.5f - o->ry);
    o->sb_x1 = (int)ceilf((float)f->crop_x1 - 0.5f + o->rx);  o->sb_y1 = (int)ceilf((float)f->crop_y1 - 0.5f + o->ry);
    // n_tiles = floor((extent + 16) / 16), integrators/sampler.jl:14-20
    o->tiles_x = (int)floorf(((float)(o->sb_x1 - o->sb_x0) + 16.0f) / 16.0f);
    o->tiles_y = (int)floorf(((float)(o->sb_y1 - o->sb_y0) + 16.0f) / 16.0f);
    o->width = f->crop_x1 - f->crop_x0 + 1; o->height = f->crop_y1 - f->crop_y0 + 1;
    TR_CUDA(c, table_buf->ensure(256 * sizeof(float)));
    TR_CUDA(c, cudaMemcpyAsync(table_buf->p, f->filter_table, 256 * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    TR_CUDA(c, cudaStreamSynchronize(c->stream));
    o->table = table_buf->as<float>();
    return 0;
}

// ------------------------------------------------------------------ ray queries
static int launch_intersect(trace_ctx* c, const float4* ro, const float4* rd, int64_t n, float4* hits) {
    int* err = ctx_icounters(c) + IC_ERROR;
    unsigned long long* cnt = ctx_stats64(c) + ST_NODES;
    const int grid = (int)std::min<int64_t>((n + 127) / 128, (int64_t)persistent_grid(c, 16));
    if (c->time_kernels) cudaEventRecord(c->evk0, c->stream);
    const DeviceScene sc = hit_launch_scene(c, c->scene);
    trav_dispatch(c, [&](auto S, auto C_, auto W) {
        constexpr int s = decltype(S)::value, w = decltype(W)::value;
        constexpr bool cn = decltype(C_)::value;
        auto k = k_intersect<s, cn, w, false>;
        if constexpr (shadow_walk_capable<s, cn, w>) if (sc.shadow_pairs) k = k_intersect<s, cn, w, true>;
        k<<<std::min(grid, occupancy_grid(c, k, 128)), 128, 0, c->stream>>>(sc, ro, rd, n, hits, cnt, err);
    });
    if (c->time_kernels) cudaEventRecord(c->evk1, c->stream);
    TR_CUDA(c, cudaGetLastError());
    c->stats.kernel_launches++;
    return 0;
}
static int launch_occluded(trace_ctx* c, const float4* ro, const float4* rd, int64_t n, uint8_t* out) {
    int* err = ctx_icounters(c) + IC_ERROR;
    unsigned long long* cnt = ctx_stats64(c) + ST_NODES;
    const int grid = (int)std::min<int64_t>((n + 127) / 128, (int64_t)persistent_grid(c, 16));
    if (c->time_kernels) cudaEventRecord(c->evk0, c->stream);
    const DeviceScene sc = shadow_launch_scene(c, c->scene);
    trav_dispatch(c, [&](auto S, auto C_, auto W) {
        constexpr int s = decltype(S)::value, w = decltype(W)::value;
        constexpr bool cn = decltype(C_)::value;
        auto k = k_occluded<s, cn, w, false>;
        if constexpr (shadow_walk_capable<s, cn, w>) if (sc.shadow_pairs) k = k_occluded<s, cn, w, true>;
        k<<<std::min(grid, occupancy_grid(c, k, 128)), 128, 0, c->stream>>>(sc, ro, rd, n, out, cnt, err);
    });
    if (c->time_kernels) cudaEventRecord(c->evk1, c->stream);
    TR_CUDA(c, cudaGetLastError());
    c->stats.kernel_launches++;
    return 0;
}

__global__ void k_add_stat(unsigned long long* stats, int slot, unsigned long long v) { stats[slot] += v; }

static int finish_query(trace_ctx* c, int stat_slot, int64_t n, bool is_shadow) {
    k_add_stat<<<1, 1, 0, c->stream>>>(ctx_stats64(c), stat_slot, (unsigned long long)n);
    TR_CUDA(c, cudaMemcpyAsync(c->h_flags, ctx_icounters(c) + IC_OVERFLOW, 2 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(c, cudaStreamSynchronize(c->stream));
    if (c->time_kernels) {
        float ms = 0.0f;
        cudaEventElapsedTime(&ms, c->evk0, c->evk1);
        if (is_shadow) { c->stats.ms_shadow += ms; c->stats.shadow_launches++; c->stats.ms_kind[TRACE_K_SHADOW] += ms; c->stats.launches_kind[TRACE_K_SHADOW]++; }
        else { c->stats.ms_extend += ms; c->stats.extend_launches++; c->stats.ms_kind[TRACE_K_EXTEND] += ms; c->stats.launches_kind[TRACE_K_EXTEND]++; }
    }
    if (c->h_flags[1]) {
        cudaMemsetAsync(ctx_icounters(c) + IC_ERROR, 0, sizeof(int), c->stream);
        return c->fail("traversal stack overflow (more than 64 pending nodes; the reference would throw a BoundsError, bvh.jl:222)");
    }
    return 0;
}

extern "C" int trace_intersect_device(trace_ctx* c, const void* ro, const void* rd, int64_t n, void* hits) {
    if (!c) return 1;
    cudaSetDevice(c->device);
    if (!c->have_scene) return c->fail("no scene uploaded");
    if (n <= 0) return 0;
    if (launch_intersect(c, (const float4*)ro, (const float4*)rd, n, (float4*)hits)) return 1;
    return finish_query(c, ST_RAYS_EXTEND, n, false);
}
extern "C" int trace_occluded_device(trace_ctx* c, const void* ro, const void* rd, int64_t n, void* out) {
    if (!c) return 1;
    cudaSetDevice(c->device);
    if (!c->have_scene) return c->fail("no scene uploaded");
    if (n <= 0) return 0;
    if (launch_occluded(c, (const float4*)ro, (const float4*)rd, n, (uint8_t*)out)) return 1;
    return finish_query(c, ST_RAYS_SHADOW, n, true);
}

static int stage_rays(trace_ctx* c, const float* o, const float* d, const float* tmax, int64_t n) {
    std::vector<float4> ho((size_t)n), hd((size_t)n);
    for (int64_t i = 0; i < n; ++i) {
        ho[i] = make_float4(o[3 * i], o[3 * i + 1], o[3 * i + 2], tmax ? tmax[i] : INFINITY);
        hd[i] = make_float4(d[3 * i], d[3 * i + 1], d[3 * i + 2], 0.0f);
    }
    TR_CUDA(c, c->b_query[0].ensure((size_t)n * sizeof(float4)));
    TR_CUDA(c, c->b_query[1].ensure((size_t)n * sizeof(float4)));
    TR_CUDA(c, cudaMemcpyAsync(c->b_query[0].p, ho.data(), (size_t)n * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
    TR_CUDA(c, cudaMemcpyAsync(c->b_query[1].p, hd.data(), (size_t)n * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
    TR_CUDA(c, cudaStreamSynchronize(c->stream));
    return 0;
}

extern "C" int trace_intersect(trace_ctx* c, const float* o, const float* d, float* tmax, int64_t n, uint32_t* prim_out,
                               float* b0b1) {
    if (!c) return 1;
    cudaSetDevice(c->device);
    if (!c->have_scene) return c->fail("no scene uploaded");
    if (n <= 0) return 0;
    if (!o || !d || !tmax || !prim_out) return c->fail("trace_intersect: null buffer");
    if (stage_rays(c, o, d, tmax, n)) return 1;
    TR_CUDA(c, c->b_query[2].ensure((size_t)n * sizeof(float4)));
    if (trace_intersect_device(c, c->b_query[0].p, c->b_query[1].p, n, c->b_query[2].p)) return 1;
    std::vector<float4> hh((size_t)n);
    TR_CUDA(c, cudaMemcpyAsync(hh.data(), c->b_query[2].p, (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(c, cudaStreamSynchronize(c->stream));
    for (int64_t i = 0; i < n; ++i) {
        uint32_t p; memcpy(&p, &hh[i].y, 4);
        prim_out[i] = p;
        if (p) tmax[i] = hh[i].x;
        if (b0b1) { b0b1[2 * i] = p ? hh[i].z : 0.0f; b0b1[2 * i + 1] = p ? hh[i].w : 0.0f; }
    }
    return 0;
}

extern "C" int trace_occluded(trace_ctx* c, const float* o, const float* d, const float* tmax, int64_t n, uint8_t* out) {
    if (!c) return 1;
    cudaSetDevice(c->device);
    if (!c->have_scene) return c->fail("no scene uploaded");
    if (n <= 0) return 0;
    if (!o || !d || !out) return c->fail("trace_occluded: null buffer");
    if (stage_rays(c, o, d, tmax, n)) return 1;
    TR_CUDA(c, c->b_query[2].ensure((size_t)n));
    if (trace_occluded_device(c, c->b_query[0].p, c->b_query[1].p, n, c->b_query[2].p)) return 1;
    TR_CUDA(c, cudaMemcpyAsync(out, c->b_query[2].p, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(c, cudaStreamSynchronize(c->stream));
    return 0;
}

// ------------------------------------------------------------------ Whitted entry points (kernels in whitted.cu)
extern "C" int trace_render_whitted_device(trace_ctx* c, const trace_camera* cam, const trace_film_desc* film, int spp,
                                           int max_depth, uint64_t seed, void* film_dev) {
    if (!c) return 1;
    cudaSetDevice(c->device);
    if (!c->have_scene) return c->fail("no scene uploaded");
    if (!cam || !film || !film_dev) return c->fail("trace_render_whitted: null argument");
    if (spp < 1 || max_depth < 1 || max_depth > TR_MAX_DEPTH) return c->fail("trace_render_whitted: spp must be >= 1 and max_depth in [1, %d]", TR_MAX_DEPTH);
    return whitted_render_device(c, cam, film, spp, max_depth, seed, (float*)film_dev);
}

extern "C" int trace_render_whitted(trace_ctx* c, const trace_camera* cam, const trace_film_desc* film, int spp, int max_depth,
                                    uint64_t seed, float* film_xyzw) {
    if (!c) return 1;
    cudaSetDevice(c->device);
    if (!cam || !film) return c->fail("trace_render_whitted: null argument");
    const size_t w = (size_t)(film->crop_x1 - film->crop_x0 + 1), h = (size_t)(film->crop_y1 - film->crop_y0 + 1);
    // the part of the film this rank delivers (all of it on one GPU; see trace_comm_init for the multi-rank modes)
    long long p0 = 0, p1 = 0;
    whitted_film_range(c, (long long)(w * h), &p0, &p1);
    if (p1 > p0 && !film_xyzw) return c->fail("trace_render_whitted: null film");
    const size_t bytes = w * h * 4 * sizeof(float), off = (size_t)p0 * 4 * sizeof(float), part = (size_t)(p1 - p0) * 4 * sizeof(float);
    TR_CUDA(c, c->b_misc[7].ensure(bytes));
    char* dev = c->b_misc[7].as<char>();
    // the caller's film is only needed by the final merge: upload it on the copy stream while the render runs
    if (part) {
        TR_CUDA(c, cudaEventRecord(c->ev_copy, c->stream));
        TR_CUDA(c, cudaStreamWaitEvent(c->copy_stream, c->ev_copy, 0));
        TR_CUDA(c, cudaMemcpyAsync(dev + off, (const char*)film_xyzw + off, part, cudaMemcpyHostToDevice, c->copy_stream));
        TR_CUDA(c, cudaEventRecord(c->ev_copy, c->copy_stream));
        c->film_upload_pending = true;
    }
    const int rc = trace_render_whitted_device(c, cam, film, spp, max_depth, seed, dev);
    if (c->film_upload_pending) { cudaStreamWaitEvent(c->stream, c->ev_copy, 0); c->film_upload_pending = false; }
    if (rc) { cudaStreamSynchronize(c->stream); return 1; }
    if (part) TR_CUDA(c, cudaMemcpyAsync((char*)film_xyzw + off, dev + off, part, cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(c, cudaStreamSynchronize(c->stream));
    return 0;
}
