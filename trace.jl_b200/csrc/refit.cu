// refit.cu — trace_scene_refit[_device] and trace_scene_copy_nodes (include/trace_cuda.h): new triangle vertices for
// the uploaded scene, with every box recomputed on the GPU over the uploaded tree's unchanged topology.
//
// The result is the scene trace_scene_upload would build from the same nodes / primitives with the new vertices and
// recomputed boxes:
//   triangle record  new p0 p1 p2; degenerate bit (30) decided again with the upload's unfused test; every other tag bit,
//                    the material and `original` kept; new normals only where the triangle has them (TRACE_TRI_HAS_NORMALS);
//   leaf box         Julia min / max (-0.0 < +0.0) union of its primitives' bounds: a triangle's three vertices, a
//                    sphere's caller-supplied bound; a zero-primitive leaf keeps its uploaded box (and its NaN box in
//                    the pair record) and contributes nothing to its parent;
//   interior box     Julia min / max union of its children's boxes (a node whose subtree holds no primitive keeps its box);
//   scene_scale      from the new root box, with the upload's rule.
// Min / max are exact, so the boxes do not depend on the order in which the climbing threads arrive: two refits with
// the same input are bit-identical.  NaN input is refused before any scene buffer is written: every writing kernel
// checks the validation pass's flag.
#include <chrono>
#include <cmath>
#include <cstring>

#include "context.hpp"
#include "traverse.cuh"

namespace {

// topology (after the upload's pair numbering, upload_device.cu): parents, each node's slot in its parent's pair record, the leaf list (leaf i is number i - pair_of[i])
__global__ void refit_topology(const float4* __restrict__ nodes, int64_t n, const uint32_t* __restrict__ pair_of,
                               int32_t* __restrict__ parent, uint32_t* __restrict__ up, uint32_t* __restrict__ leaves) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (i == 0) { parent[0] = -1; up[0] = 0u; }
    const float4 b = nodes[2 * i + 1];
    if (tr_node_leaf(__float_as_uint(b.w))) { leaves[i - pair_of[i]] = (uint32_t)i; return; }
    const uint32_t q = pair_of[i], second = __float_as_uint(b.z);
    parent[i + 1] = (int32_t)i; up[i + 1] = 2u * q;
    parent[second] = (int32_t)i; up[second] = 2u * q + 1u;
}

// 1. NaN anywhere in the input
__global__ void refit_validate(const float* __restrict__ v, int64_t n, uint32_t* status) {
    bool nan = false;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        nan |= v[i] != v[i];
    if (__any_sync(0xFFFFFFFFu, nan) && (threadIdx.x & 31) == 0) atomicOr(status, 1u);
}

// 2. one thread per primitive slot: new vertices (and normals) into the BVH-ordered records, degenerate bit again
__global__ void refit_scatter(const float* __restrict__ v, const float* __restrict__ nrm, int64_t n_prims,
                              const uint32_t* __restrict__ slot_tri, const uint32_t* __restrict__ status,
                              float4* __restrict__ prims, float4* __restrict__ tnorm) {
    const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= n_prims || *status) return;
    const float4 A = prims[3 * s];
    uint32_t tag = __float_as_uint(A.w);
    if (tag & TR_PRIM_SPHERE_BIT) return;
    const size_t t = slot_tri[s];
    const float* p = v + 9 * t;
    const float3 p0 = f3(p[0], p[1], p[2]), p1 = f3(p[3], p[4], p[5]), p2 = f3(p[6], p[7], p[8]);
    tag = tri_degenerate(p0, p1, p2) ? (tag | TR_PRIM_DEGENERATE_BIT) : (tag & ~TR_PRIM_DEGENERATE_BIT);
    const float mat = prims[3 * s + 1].w, orig = prims[3 * s + 2].w;
    prims[3 * s] = f4(p0, __uint_as_float(tag));
    prims[3 * s + 1] = f4(p1, mat);
    prims[3 * s + 2] = f4(p2, orig);
    if (!nrm) return;
    const float4 N0 = tnorm[3 * s];
    if (!(__float_as_uint(N0.w) & TRACE_TRI_HAS_NORMALS)) return;
    const float* q = nrm + 9 * t;
    tnorm[3 * s] = make_float4(q[0], q[1], q[2], N0.w);
    tnorm[3 * s + 1] = make_float4(q[3], q[4], q[5], tnorm[3 * s + 1].w);
    tnorm[3 * s + 2] = make_float4(q[6], q[7], q[8], tnorm[3 * s + 2].w);
}

// a node's box into its node record (offset / meta words untouched) and into its half of the parent's pair record
// (reference and split-axis words untouched)
__device__ __forceinline__ void put_box(float4* nodes, float4* pairs, const uint32_t* up, int64_t v, const float lo[3],
                                        const float hi[3]) {
    const float4 a = make_float4(lo[0], lo[1], lo[2], hi[0]);
    const float2 b = make_float2(hi[1], hi[2]);
    nodes[2 * v] = a;
    *reinterpret_cast<float2*>(&nodes[2 * v + 1]) = b;
    if (v == 0) return;
    const uint32_t u = up[v];
    float4* q = pairs + 4 * (size_t)(u >> 1) + 2 * (u & 1u);
    q[0] = a;
    *reinterpret_cast<float2*>(&q[1]) = b;
}

// 3. one thread per leaf: the leaf's box, then climb while it is the second to arrive (as lbvh_bottom_up)
__global__ void refit_climb(const float4* __restrict__ prims, const float* __restrict__ sphere_bounds, int64_t n_leaves,
                            const uint32_t* __restrict__ leaves, const int32_t* __restrict__ parent,
                            const uint32_t* __restrict__ up, uint32_t* arrive, uint8_t* empty,
                            const uint32_t* __restrict__ status, float4* nodes, float4* pairs) {
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= n_leaves || *status) return;
    int64_t v = leaves[k];
    float lo[3] = {TR_INF, TR_INF, TR_INF}, hi[3] = {-TR_INF, -TR_INF, -TR_INF};
    bool e;
    {
        const float4 b = nodes[2 * v + 1];
        const uint32_t first = __float_as_uint(b.z), cnt = tr_node_count(__float_as_uint(b.w));
        for (uint32_t j = 0; j < cnt; ++j) {
            const int64_t s = first + j;
            const float4 A = prims[3 * s];
            const uint32_t tag = __float_as_uint(A.w);
            if (tag & TR_PRIM_SPHERE_BIT) {
                const float* sb = sphere_bounds + 6 * (size_t)(tag & TR_PRIM_INDEX_MASK);
                for (int c = 0; c < 3; ++c) { lo[c] = jl_min(lo[c], sb[c]); hi[c] = jl_max(hi[c], sb[3 + c]); }
            } else {
                tri_box(xyz(A), xyz(prims[3 * s + 1]), xyz(prims[3 * s + 2]), lo, hi);
            }
        }
        // (+inf, -inf) is the identity of the union, so an empty subtree's registers never change a sibling's box
        e = cnt == 0;
        empty[v] = e;
        if (!e) put_box(nodes, pairs, up, v, lo, hi);
    }
    for (;;) {
        const int32_t p = parent[v];
        if (p < 0) break;
        const uint32_t u = up[v];
        __threadfence();
        if (atomicAdd(&arrive[u >> 1], 1u) == 0) return;          // the sibling's thread continues
        __threadfence();
        const int64_t sib = (u & 1u) ? (int64_t)p + 1 : (int64_t)__float_as_uint(__ldcg(&nodes[2 * (int64_t)p + 1]).z);
        const bool sib_empty = *(volatile const uint8_t*)&empty[sib] != 0;
        if (!sib_empty) {
            const float4 a = __ldcg(&nodes[2 * sib]);
            const float2 b = __ldcg(reinterpret_cast<const float2*>(&nodes[2 * sib + 1]));
            lo[0] = jl_min(lo[0], a.x); lo[1] = jl_min(lo[1], a.y); lo[2] = jl_min(lo[2], a.z);
            hi[0] = jl_max(hi[0], a.w); hi[1] = jl_max(hi[1], b.x); hi[2] = jl_max(hi[2], b.y);
        }
        e = e && sib_empty;
        empty[p] = e;
        if (!e) put_box(nodes, pairs, up, p, lo, hi);
        v = p;
    }
}

// ------------------------------------------------------------------ the shadow tree (api.cu, traverse.cuh traverse_shadow)
// Its pair records hold both children's boxes, so a pair's box is the union of its own two halves: one thread per
// primitive writes the primitive's vertex box into its leaf's half, then climbs while it is the second to arrive at a
// pair, writing the pair's union into the parent's half.  Same rules as above (Julia min / max, exact, deterministic)
// and as the build (bvh_gpu.cu), so a refit with unchanged vertices gives back the uploaded records.

// topology: every reference's (parent pair, slot)
__global__ void shadow_topology(const float4* __restrict__ pairs, int64_t n_pairs, uint32_t* __restrict__ up_pair,
                                uint32_t* __restrict__ up_prim) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n_pairs) return;
    for (uint32_t k = 0; k < 2; ++k) {
        const uint32_t ref = __float_as_uint(pairs[4 * i + 2 * k + 1].z), u = 2u * (uint32_t)i + k;
        if (ref & TR_REF_LEAF) up_prim[ref & TR_REF_INDEX_MASK] = u;
        else up_pair[ref] = u;
    }
}

__device__ __forceinline__ void put_half(float4* pairs, uint32_t u, const float lo[3], const float hi[3]) {
    float4* q = pairs + 4 * (size_t)(u >> 1) + 2 * (u & 1u);
    q[0] = make_float4(lo[0], lo[1], lo[2], hi[0]);
    *reinterpret_cast<float2*>(&q[1]) = make_float2(hi[1], hi[2]);
}

__global__ void shadow_climb(const float4* __restrict__ prims, int64_t n_prims, const uint32_t* __restrict__ up_pair,
                             const uint32_t* __restrict__ up_prim, uint32_t* arrive, const uint32_t* __restrict__ status,
                             float4* pairs) {
    const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= n_prims || *status) return;
    float lo[3] = {TR_INF, TR_INF, TR_INF}, hi[3] = {-TR_INF, -TR_INF, -TR_INF};
    tri_box(xyz(prims[3 * s]), xyz(prims[3 * s + 1]), xyz(prims[3 * s + 2]), lo, hi);
    uint32_t u = up_prim[s];
    put_half(pairs, u, lo, hi);
    for (;;) {
        const uint32_t p = u >> 1;
        __threadfence();
        if (atomicAdd(&arrive[p], 1u) == 0) return;               // the sibling's thread continues
        __threadfence();
        const float4 a0 = __ldcg(&pairs[4 * (size_t)p]), a1 = __ldcg(&pairs[4 * (size_t)p + 1]);
        const float4 b0 = __ldcg(&pairs[4 * (size_t)p + 2]), b1 = __ldcg(&pairs[4 * (size_t)p + 3]);
        lo[0] = jl_min(a0.x, b0.x); lo[1] = jl_min(a0.y, b0.y); lo[2] = jl_min(a0.z, b0.z);
        hi[0] = jl_max(a0.w, b0.w); hi[1] = jl_max(a1.x, b1.x); hi[2] = jl_max(a1.y, b1.y);
        u = up_pair[p];
        if (u == ~0u) return;                                      // the root: pair 0 has no parent half
        put_half(pairs, u, lo, hi);
    }
}

// first refit after an upload: parents, pair slots and leaves from b_nodes, the slot -> triangle map from the host (or,
// after a device mesh upload, the one it left on the device)
int derive_topology(trace_ctx* c) {
    auto& R = c->refit;
    const int64_t n = c->scene.n_nodes, n_prims = c->scene.n_prims, n_leaves = n - R.n_pairs;
    const size_t scan_bytes = pair_scan_bytes(n, c->stream);
    if (!scan_bytes) return c->fail("scene refit: cannot size the pair scan");
    Carve k;
    const size_t o_parent = k.take(n * 4), o_up = k.take(n * 4), o_pair = k.take(n * 4), o_leaves = k.take(n_leaves * 4),
                 o_empty = k.take(n), o_arrive = k.take(R.n_pairs * 4), o_tri = k.take(R.slot_tri_on_device ? 0 : n_prims * 4),
                 o_status = k.take(16), o_scan = k.take(scan_bytes);
    TR_CUDA(c, R.topo.ensure(k.used));
    char* base = R.topo.as<char>();
    R.parent = (int32_t*)(base + o_parent); R.up = (uint32_t*)(base + o_up); R.pair_of = (uint32_t*)(base + o_pair);
    R.leaves = (uint32_t*)(base + o_leaves); R.empty = (uint8_t*)(base + o_empty); R.arrive = (uint32_t*)(base + o_arrive);
    R.slot_tri = R.slot_tri_on_device ? R.slot_tri_dev.as<uint32_t>() : (uint32_t*)(base + o_tri);
    R.status = (uint32_t*)(base + o_status);
    const int T = 256;
    TR_CUDA(c, pair_numbering(c->stream, c->scene.nodes, n, R.up, R.pair_of, base + o_scan, scan_bytes));   // (`up` holds the flags until the scan)
    refit_topology<<<blocks_for(n, T), T, 0, c->stream>>>(c->scene.nodes, n, R.pair_of, R.parent, R.up, R.leaves);
    TR_CUDA(c, cudaGetLastError());
    if (n_prims && !R.slot_tri_on_device)
        TR_CUDA(c, cudaMemcpyAsync(R.slot_tri, R.tri_index.data(), (size_t)n_prims * 4, cudaMemcpyHostToDevice, c->stream));
    TR_CUDA(c, cudaStreamSynchronize(c->stream));       // (tri_index is pageable host memory)
    R.topo_ready = true;
    return 0;
}

// first refit after an upload that built a shadow tree: its parents, from the pair records
int derive_shadow_topology(trace_ctx* c) {
    auto& R = c->refit;
    const int64_t n_prims = c->scene.n_prims, n_pairs = n_prims - 1;
    Carve k;
    const size_t o_up_pair = k.take(n_pairs * 4), o_up_prim = k.take(n_prims * 4), o_arrive = k.take(n_pairs * 4);
    TR_CUDA(c, R.shadow_topo.ensure(k.used));
    char* base = R.shadow_topo.as<char>();
    R.shadow_up_pair = (uint32_t*)(base + o_up_pair); R.shadow_up_prim = (uint32_t*)(base + o_up_prim);
    R.shadow_arrive = (uint32_t*)(base + o_arrive);
    TR_CUDA(c, cudaMemsetAsync(R.shadow_up_pair, 0xFF, n_pairs * 4, c->stream));
    shadow_topology<<<blocks_for(n_pairs, 256), 256, 0, c->stream>>>(c->scene.shadow_pairs, n_pairs, R.shadow_up_pair, R.shadow_up_prim);
    TR_CUDA(c, cudaGetLastError());
    R.shadow_topo_ready = true;
    return 0;
}

int check_args(trace_ctx* c, int64_t n_tris, const void* v, int64_t n_spheres, const float* sb) {
    if (!c->have_scene) return c->fail("scene refit: no scene uploaded");
    const auto& R = c->refit;
    if (n_tris != R.n_tris) return c->fail("scene refit: %lld triangles given, the uploaded scene has %lld", (long long)n_tris, (long long)R.n_tris);
    if (n_tris > 0 && !v) return c->fail("scene refit: null vertex buffer");
    if (R.n_spheres > 0) {
        if (!sb) return c->fail("scene refit: the scene holds %lld spheres and no sphere bounds were given", (long long)R.n_spheres);
        if (n_spheres != R.n_spheres) return c->fail("scene refit: %lld sphere bounds given, the uploaded scene has %lld spheres", (long long)n_spheres, (long long)R.n_spheres);
        for (int64_t i = 0; i < 6 * n_spheres; ++i)
            if (std::isnan(sb[i])) return c->fail("scene refit: sphere %lld has a NaN bound", (long long)(i / 6));
    }
    return 0;
}

// The one implementation: v / nrm are device pointers, or (host_input) host pointers staged first.
int refit_run(trace_ctx* c, int64_t n_tris, const float* v, const float* nrm, bool host_input, int64_t n_spheres,
              const float* sb) {
    cudaSetDevice(c->device);
    if (check_args(c, n_tris, v, n_spheres, sb)) return 1;
    if (c->scene.n_nodes == 0) return 0;                   // an empty scene: no triangle, no box
    auto& R = c->refit;
    PhaseTimer ph;
    ph.on = getenv("TRACE_BVH_PROFILE") != nullptr;
    const auto t0 = std::chrono::steady_clock::now();
    if (ctx_drain(c)) return 1;
    sppm_end_session(c);
    ph.mark(c->stream, nullptr);
    if (!R.topo_ready) {
        if (derive_topology(c)) return 1;
        ph.mark(c->stream, "topology");
    }
    const size_t vbytes = (size_t)n_tris * 9 * sizeof(float);
    if (host_input && n_tris > 0) {
        TR_CUDA(c, R.stage.ensure(nrm ? 2 * vbytes : vbytes));
        TR_CUDA(c, cudaMemcpyAsync(R.stage.p, v, vbytes, cudaMemcpyHostToDevice, c->stream));
        if (nrm) TR_CUDA(c, cudaMemcpyAsync(R.stage.as<char>() + vbytes, nrm, vbytes, cudaMemcpyHostToDevice, c->stream));
        v = R.stage.as<float>();
        nrm = nrm ? reinterpret_cast<const float*>(R.stage.as<char>() + vbytes) : nullptr;
        ph.mark(c->stream, "stage");
    }
    if (R.n_spheres > 0) {
        TR_CUDA(c, R.sphere_bounds.ensure((size_t)n_spheres * 6 * sizeof(float)));
        TR_CUDA(c, cudaMemcpyAsync(R.sphere_bounds.p, sb, (size_t)n_spheres * 6 * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    }
    const int64_t n_nodes = c->scene.n_nodes, n_prims = c->scene.n_prims, n_leaves = n_nodes - R.n_pairs;
    float4* nodes = c->b_nodes.as<float4>();
    TR_CUDA(c, cudaMemsetAsync(R.status, 0, 16, c->stream));
    if (R.n_pairs) TR_CUDA(c, cudaMemsetAsync(R.arrive, 0, (size_t)R.n_pairs * 4, c->stream));
    const int T = 256;
    if (n_tris > 0) {
        const int64_t nf = 9 * n_tris;
        const unsigned grid = (unsigned)std::min<int64_t>(blocks_for(nf, T), (int64_t)c->num_sms * 8);
        refit_validate<<<grid, T, 0, c->stream>>>(v, nf, R.status);
        if (nrm) refit_validate<<<grid, T, 0, c->stream>>>(nrm, nf, R.status);
    }
    ph.mark(c->stream, "validate");
    if (n_prims > 0)
        refit_scatter<<<blocks_for(n_prims, T), T, 0, c->stream>>>(v, nrm, n_prims, R.slot_tri, R.status, c->b_prims.as<float4>(),
                                                                   c->b_tnorm.as<float4>());
    ph.mark(c->stream, "scatter");
    if (n_leaves > 0)
        refit_climb<<<blocks_for(n_leaves, T), T, 0, c->stream>>>(c->b_prims.as<float4>(), R.sphere_bounds.as<float>(), n_leaves,
                                                                  R.leaves, R.parent, R.up, R.arrive, R.empty, R.status, nodes,
                                                                  c->b_pairs.as<float4>());
    TR_CUDA(c, cudaGetLastError());
    ph.mark(c->stream, "climb");
    if (c->scene.shadow_pairs) {                           // the shadow tree: same primitives, its own topology
        if (!R.shadow_topo_ready && derive_shadow_topology(c)) return 1;
        TR_CUDA(c, cudaMemsetAsync(R.shadow_arrive, 0, (size_t)(n_prims - 1) * 4, c->stream));
        shadow_climb<<<blocks_for(n_prims, T), T, 0, c->stream>>>(c->b_prims.as<float4>(), n_prims, R.shadow_up_pair,
                                                                  R.shadow_up_prim, R.shadow_arrive, R.status,
                                                                  c->b_shadow.as<float4>());
        TR_CUDA(c, cudaGetLastError());
        ph.mark(c->stream, "shadow tree");
    }
    uint32_t nan = 0;
    float4 root[2] = {};
    TR_CUDA(c, cudaMemcpyAsync(&nan, R.status, 4, cudaMemcpyDeviceToHost, c->stream));
    if (n_nodes > 0) TR_CUDA(c, cudaMemcpyAsync(root, nodes, sizeof(root), cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(c, cudaStreamSynchronize(c->stream));
    ph.mark(c->stream, "readback");
    if (nan) return c->fail("scene refit: NaN in the new vertices or normals (the scene is unchanged)");
    // a composed scene without a shadow tree left the base's and the meshes' shadow pairs with the old boxes: later
    // attaches get none while one of those parts is in the scene
    if (c->base.moved && !c->scene.shadow_pairs) {
        if (c->base.shadow_depth > 1) c->base.shadow_depth = 0;
        for (auto& sl : c->slots) if (sl.shadow_depth > 1) sl.shadow_depth = 0;
    }
    if (n_nodes > 0) {                                     // the upload's rule (api.cu)
        const float b[6] = {root[0].x, root[0].y, root[0].z, root[0].w, root[1].x, root[1].y};
        float scale = 0.0f;
        for (int k = 0; k < 6; ++k) if (std::isfinite(fabsf(b[k]))) scale = fmaxf(scale, fabsf(b[k]));
        c->scene.scene_scale = scale;
    }
    if (ph.on) {
        cudaEventSynchronize(ph.ev[ph.n - 1]);
        char head[160];
        snprintf(head, sizeof(head), "scene refit: %lld triangles, %lld nodes, %s input", (long long)n_tris, (long long)n_nodes,
                 host_input ? "host" : "device");
        ph.print(head, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
    }
    return 0;
}

}  // namespace

extern "C" int trace_scene_refit(trace_ctx* c, int64_t n_tris, const float* tri_vertices, const float* tri_normals,
                                 int64_t n_spheres, const float* sphere_bounds) {
    if (!c) return 1;
    return refit_run(c, n_tris, tri_vertices, tri_normals, true, n_spheres, sphere_bounds);
}

extern "C" int trace_scene_refit_device(trace_ctx* c, int64_t n_tris, const void* tri_vertices_device,
                                        const void* tri_normals_device, int64_t n_spheres, const float* sphere_bounds) {
    if (!c) return 1;
    return refit_run(c, n_tris, (const float*)tri_vertices_device, (const float*)tri_normals_device, false, n_spheres,
                     sphere_bounds);
}

extern "C" int trace_scene_copy_nodes(trace_ctx* c, trace_bvh_node* out) {
    if (!c) return 1;
    cudaSetDevice(c->device);
    if (!c->have_scene) return c->fail("no scene uploaded");
    const int64_t n = c->scene.n_nodes;
    if (n > 0 && !out) return c->fail("trace_scene_copy_nodes: null buffer");
    std::vector<float4> h((size_t)n * 2);
    if (n > 0) {
        TR_CUDA(c, cudaMemcpyAsync(h.data(), c->b_nodes.p, h.size() * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
        TR_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    for (int64_t i = 0; i < n; ++i) {
        const float4 a = h[2 * i], b = h[2 * i + 1];
        trace_bvh_node& o = out[i];
        o.bmin[0] = a.x; o.bmin[1] = a.y; o.bmin[2] = a.z; o.bmax[0] = a.w; o.bmax[1] = b.x; o.bmax[2] = b.y;
        memcpy(&o.offset, &b.z, 4); memcpy(&o.meta, &b.w, 4);
        o.meta &= ~TR_NODE_SPHERE_BELOW;                   // the device-only "sphere below" bit (api.cu)
    }
    return 0;
}
