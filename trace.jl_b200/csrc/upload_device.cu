// upload_device.cu — trace_scene_upload_mesh_device (include/trace_cuda.h): a triangle-only scene whose per-triangle
// arrays are in device memory, with its tree built and every scene buffer written on the GPU; and the pair records of
// every upload (ctx_pack_pairs, also run by trace_scene_upload once its nodes and primitives are on the device).
//
// The result is the scene trace_scene_upload (api.cu) builds from the LBVH of the triangles' Julia min / max boxes
// and prims[k] = {TRIANGLE, order[k], material[order[k]], order[k]}.  The steps, all on the context's stream:
//   validate   NaN normals, material indices >= n_materials           } lbvh_mesh_build (bvh_gpu.cu): into the LBVH's
//   bounds     triangle boxes from the [n][3][3] vertices (NaN: refused) } status block, read back with the build's
//   build      keys, sort, hierarchy, bottom-up boxes                   } status before any scene buffer is written
//   emit       the preorder node records straight into b_nodes (trace_bvh_node has the layout of two float4);
//   scatter    one thread per slot: the primitive and normal records, degenerate bit as the host upload decides it;
//   pairs      ctx_pack_pairs: the preorder pair numbering (a scan of "is interior"), then one thread per node: the
//              pair record of an interior node, the last-of-leaf bit of a leaf's last primitive;
//   readback   the root box (scene_scale);
//   shadow     the shadow tree over the new primitive records (the host upload's tail, ctx_commit_scene).
#include <chrono>
#include <cmath>
#include <cstring>

#include <cub/device/device_scan.cuh>

#include "context.hpp"
#include "traverse.cuh"

namespace {

// scatter: slot s holds triangle order[s] (trace_scene_upload's per-primitive loop, triangles only)
__global__ void upload_scatter(const float* __restrict__ v, const float* __restrict__ nrm, const uint8_t* __restrict__ flg,
                               const uint32_t* __restrict__ mat, const uint32_t* __restrict__ order, int64_t n,
                               float4* __restrict__ prims, float4* __restrict__ tnorm) {
    const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= n) return;
    const uint32_t t = order[s];
    const float* p = v + 9 * (size_t)t;
    const float3 p0 = f3(p[0], p[1], p[2]), p1 = f3(p[3], p[4], p[5]), p2 = f3(p[6], p[7], p[8]);
    const uint32_t tag = tri_degenerate(p0, p1, p2) ? TR_PRIM_DEGENERATE_BIT : 0u;
    prims[3 * s] = f4(p0, __uint_as_float(tag));
    prims[3 * s + 1] = f4(p1, __uint_as_float(mat ? mat[t] : 0u));
    prims[3 * s + 2] = f4(p2, __uint_as_float(t));
    uint32_t flags = flg ? flg[t] : 0u;
    if (!nrm) flags &= ~(uint32_t)TRACE_TRI_HAS_NORMALS;
    float4 N0 = make_float4(0.0f, 0.0f, 0.0f, __uint_as_float(flags)), N1 = make_float4(0.0f, 0.0f, 0.0f, 0.0f), N2 = N1;
    if (flags & TRACE_TRI_HAS_NORMALS) {
        const float* q = nrm + 9 * (size_t)t;
        N0.x = q[0]; N0.y = q[1]; N0.z = q[2]; N1.x = q[3]; N1.y = q[4]; N1.z = q[5]; N2.x = q[6]; N2.y = q[7]; N2.z = q[8];
    }
    tnorm[3 * s] = N0;
    tnorm[3 * s + 1] = N1;
    tnorm[3 * s + 2] = N2;
}

// 1 for an interior node (scanned into the preorder pair numbering)
__global__ void pair_is_interior(const float4* __restrict__ nodes, int64_t n, uint32_t* __restrict__ flag) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) flag[i] = tr_node_leaf(__float_as_uint(nodes[2 * i + 1].w)) ? 0u : 1u;
}

// pairs (traverse.cuh, the pair-node walk): one thread per node.  A leaf marks its last primitive; an interior node
// writes both children's boxes and references into its pair record, the split axis as a bit in the first half.  A
// zero-primitive leaf owns no primitive and is never entered: its box is invalid and fails every slab test in the
// reference (Q16/Q17), enforced here with a NaN box.
__global__ void upload_pairs(const float4* __restrict__ nodes, int64_t n, const uint32_t* __restrict__ pair_of,
                             float4* __restrict__ prims, float4* __restrict__ pairs) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 nb = nodes[2 * i + 1];
    const uint32_t meta = __float_as_uint(nb.w);
    if (tr_node_leaf(meta)) {
        const uint32_t cnt = tr_node_count(meta);
        if (cnt) {
            float* w = &prims[3 * (size_t)(__float_as_uint(nb.z) + cnt - 1)].w;
            *w = __uint_as_float(__float_as_uint(*w) | TR_PRIM_LAST_BIT);
        }
        return;
    }
    const int64_t kids[2] = {i + 1, (int64_t)__float_as_uint(nb.z)};
    float4* q = pairs + 4 * (size_t)pair_of[i];
    for (int k = 0; k < 2; ++k) {
        float4 a = nodes[2 * kids[k]], b = nodes[2 * kids[k] + 1];
        const uint32_t cm = __float_as_uint(b.w);
        const bool leaf = tr_node_leaf(cm);
        if (leaf && tr_node_count(cm) == 0u) { a.x = a.y = a.z = a.w = __int_as_float(0x7fc00000); b.x = b.y = a.x; }   // nanf("")
        const uint32_t below = (cm & TR_NODE_SPHERE_BELOW) ? TR_REF_SPHERE_BELOW : 0u;
        const uint32_t ref = below | (leaf ? (TR_REF_LEAF | __float_as_uint(b.z)) : pair_of[kids[k]]);
        b.z = __uint_as_float(ref);
        b.w = __uint_as_float(k == 0 ? (1u << tr_node_axis(meta)) : 0u);
        q[2 * k] = a;
        q[2 * k + 1] = b;
    }
}

int upload(trace_ctx* c, const trace_mesh_device_desc* d, int64_t* n_nodes_out) {
    const int64_t n = d->n_tris;
    if (n < 0 || n >= (1ll << 30)) return c->fail("mesh upload: n_tris must be in [0, 2^30)");
    if (n > 0 && !d->tri_vertices) return c->fail("mesh upload: null vertex array");
    std::vector<DeviceMaterial> mats;
    std::vector<DeviceLight> lights;
    if (ctx_pack_materials(c, d->n_materials, d->materials, mats) || ctx_pack_lights(c, d->n_lights, d->lights, lights)) return 1;
    const int m = d->max_node_primitives < 1 ? 1 : (d->max_node_primitives < 255 ? d->max_node_primitives : 255);
    PhaseTimer ph;
    ph.on = getenv("TRACE_BVH_PROFILE") != nullptr;
    const auto t0 = std::chrono::steady_clock::now();
    if (ctx_drain(c)) return 1;
    cudaStream_t s = c->stream;
    ph.mark(s, nullptr);
    const float* v = static_cast<const float*>(d->tri_vertices);
    const float* nrm = static_cast<const float*>(d->tri_normals);
    int64_t n_nodes = 0;
    if (n == 0) {                                          // the empty scene, as trace_scene_upload stores it
        if (ctx_put(c, c->b_nodes, nullptr, 0) || ctx_put(c, c->b_pairs, nullptr, 0) || ctx_put(c, c->b_prims, nullptr, 0) ||
            ctx_put(c, c->b_tnorm, nullptr, 0))
            return 1;
    } else {
        // scratch: the LBVH build (reused by the shadow tree's), then the pair numbering's
        const int64_t nn = 2 * n - 1;
        const size_t scan_bytes = pair_scan_bytes(nn, s), lbvh_bytes = lbvh_scratch_bytes(n, s);
        if (!scan_bytes || !lbvh_bytes) return c->fail("mesh upload: cannot size the sort or the scan");
        Carve k;
        k.take(lbvh_bytes);
        const size_t o_pairs = k.take(pair_scratch_bytes(nn, scan_bytes));
        TR_CUDA(c, c->b_build.ensure(k.used));
        char* scratch = c->b_build.as<char>();
        const uint32_t* order = nullptr;
        switch (lbvh_mesh_build(s, v, nrm, static_cast<const uint32_t*>(d->tri_materials), d->n_materials, n, m, scratch, ph,
                                &n_nodes, &order)) {
            case LBVH_OK: break;
            case LBVH_NAN_BOUND: return c->fail("mesh upload: NaN in a triangle vertex (the scene is unchanged)");
            case LBVH_TOO_DEEP: return c->fail("mesh upload: the tree is deeper than 64 levels, the traversal stack (the scene is unchanged)");
            case LBVH_NAN_NORMAL: return c->fail("mesh upload: NaN in a triangle normal (the scene is unchanged)");
            case LBVH_BAD_MATERIAL: return c->fail("mesh upload: a material index is out of range (%lld materials; the scene is unchanged)", (long long)d->n_materials);
            default: return c->fail("mesh upload: CUDA error in the tree build (%s)", cudaGetErrorString(cudaGetLastError()));
        }
        // --- accepted: from here on the scene buffers are rewritten
        const int64_t n_pairs = (n_nodes - 1) / 2;       // a full binary tree
        TR_CUDA(c, c->b_nodes.ensure((size_t)n_nodes * 2 * sizeof(float4)));
        TR_CUDA(c, c->b_pairs.ensure(n_pairs ? (size_t)n_pairs * 4 * sizeof(float4) : 16));
        TR_CUDA(c, c->b_prims.ensure((size_t)n * 3 * sizeof(float4)));
        TR_CUDA(c, c->b_tnorm.ensure((size_t)n * 3 * sizeof(float4)));
        TR_CUDA(c, c->refit.slot_tri_dev.ensure((size_t)n * sizeof(uint32_t)));
        if (lbvh_mesh_emit(s, n, m, scratch, c->b_nodes.p)) return c->fail("mesh upload: CUDA error in emit");
        ph.mark(s, "emit");
        const int T = 256;
        upload_scatter<<<blocks_for(n, T), T, 0, s>>>(v, nrm, static_cast<const uint8_t*>(d->tri_flags),
                                                      static_cast<const uint32_t*>(d->tri_materials), order, n,
                                                      c->b_prims.as<float4>(), c->b_tnorm.as<float4>());
        TR_CUDA(c, cudaGetLastError());
        TR_CUDA(c, cudaMemcpyAsync(c->refit.slot_tri_dev.p, order, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToDevice, s));
        ph.mark(s, "scatter");
        if (ctx_pack_pairs(c, n_nodes, scratch + o_pairs, scan_bytes)) return 1;
        ph.mark(s, "pairs");
    }
    if (ctx_put(c, c->b_spheres, nullptr, 0) || ctx_put(c, c->b_materials, mats.data(), mats.size() * sizeof(DeviceMaterial)) ||
        ctx_put(c, c->b_lights, lights.data(), lights.size() * sizeof(DeviceLight)))
        return 1;
    float4 root[2] = {};
    if (n_nodes > 0) TR_CUDA(c, cudaMemcpyAsync(root, c->b_nodes.p, sizeof(root), cudaMemcpyDeviceToHost, s));
    TR_CUDA(c, cudaStreamSynchronize(s));                  // (the materials / lights staging vectors die at return)
    ph.mark(s, "readback");
    std::vector<uint32_t>().swap(c->refit.tri_index);
    c->refit.slot_tri_on_device = true;
    if (ctx_commit_scene(c, n_nodes, n, 0, d->n_materials, d->n_lights, n, n_nodes > 0 ? (n_nodes - 1) / 2 : 0, root,
                         c->b_build.p))
        return 1;
    ph.mark(s, "shadow-tree");
    if (n_nodes_out) *n_nodes_out = n_nodes;
    if (ph.on) {
        cudaEventSynchronize(ph.ev[ph.n - 1]);
        char head[160];
        snprintf(head, sizeof(head), "scene upload mesh device: %lld triangles, %lld nodes", (long long)n, (long long)n_nodes);
        ph.print(head, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
    }
    return 0;
}

}  // namespace

size_t pair_scan_bytes(int64_t n, cudaStream_t s) {
    size_t bytes = 0;
    if (cub::DeviceScan::ExclusiveSum(nullptr, bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)n, s) != cudaSuccess)
        return 0;
    return bytes ? bytes : 1;
}

cudaError_t pair_numbering(cudaStream_t s, const float4* nodes, int64_t n, uint32_t* flag, uint32_t* pair_of, void* tmp,
                           size_t tmp_bytes) {
    pair_is_interior<<<blocks_for(n, 256), 256, 0, s>>>(nodes, n, flag);
    const cudaError_t e = cudaGetLastError();
    return e != cudaSuccess ? e : cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, flag, pair_of, (int)n, s);
}

// ctx_pack_pairs' scratch over n nodes: the flags, the pair numbers and scan_bytes (pair_scan_bytes(n)) of scan temp
size_t pair_scratch_bytes(int64_t n, size_t scan_bytes) {
    Carve k;
    k.take(n * 4); k.take(n * 4); k.take(scan_bytes);
    return k.used;
}

// The pair records of the scene's n_nodes >= 1 preorder node records in b_nodes into b_pairs (sized for them), and the
// last-of-leaf bit of every leaf's last primitive into b_prims; `scratch`: pair_scratch_bytes(n_nodes, scan_bytes) bytes
int ctx_pack_pairs(trace_ctx* c, int64_t n_nodes, char* scratch, size_t scan_bytes) {
    Carve k;
    uint32_t* flag = reinterpret_cast<uint32_t*>(scratch + k.take(n_nodes * 4));
    uint32_t* pair_of = reinterpret_cast<uint32_t*>(scratch + k.take(n_nodes * 4));
    char* scan = scratch + k.take(scan_bytes);
    const float4* nodes = c->b_nodes.as<float4>();
    TR_CUDA(c, pair_numbering(c->stream, nodes, n_nodes, flag, pair_of, scan, scan_bytes));
    upload_pairs<<<blocks_for(n_nodes, 256), 256, 0, c->stream>>>(nodes, n_nodes, pair_of, c->b_prims.as<float4>(),
                                                                  c->b_pairs.as<float4>());
    TR_CUDA(c, cudaGetLastError());
    return 0;
}

extern "C" int trace_scene_upload_mesh_device(trace_ctx* c, const trace_mesh_device_desc* d, int64_t* n_nodes_out) {
    if (!c || !d) return 1;
    cudaSetDevice(c->device);
    return upload(c, d, n_nodes_out);
}
