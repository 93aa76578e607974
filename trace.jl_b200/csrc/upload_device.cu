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
//
// trace_scene_attach_mesh_device composes such a mesh with the scene of the last upload (the base) under a new root:
// the same steps over the mesh, with its records written after the base's and every reference shifted past them,
// then node 0, pair 0 and shadow pair 0 over the two parts (attach_root).  The first attach after an upload moves the
// base's records up one slot (attach_move_base); later ones leave the base alone.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>

#include <cub/device/device_scan.cuh>

#include "context.hpp"
#include "traverse.cuh"

namespace {

// scatter: slot s holds triangle order[s] (trace_scene_upload's per-primitive loop, triangles only) as primitive
// {TRIANGLE, tri_shift + t, mat_shift + material, prim_shift + t}; slot[s] = tri_shift + t is the refit's slot ->
// triangle map.  The shifts are the base's counts in an attach, else 0.
__global__ void upload_scatter(const float* __restrict__ v, const float* __restrict__ nrm, const uint8_t* __restrict__ flg,
                               const uint32_t* __restrict__ mat, const uint32_t* __restrict__ order, int64_t n,
                               uint32_t tri_shift, uint32_t mat_shift, uint32_t prim_shift, float4* __restrict__ prims,
                               float4* __restrict__ tnorm, uint32_t* __restrict__ slot) {
    const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= n) return;
    const uint32_t t = order[s];
    const float* p = v + 9 * (size_t)t;
    const float3 p0 = f3(p[0], p[1], p[2]), p1 = f3(p[3], p[4], p[5]), p2 = f3(p[6], p[7], p[8]);
    const uint32_t tag = tri_degenerate(p0, p1, p2) ? TR_PRIM_DEGENERATE_BIT : 0u;
    prims[3 * s] = f4(p0, __uint_as_float(tag));
    prims[3 * s + 1] = f4(p1, __uint_as_float(mat_shift + (mat ? mat[t] : 0u)));
    prims[3 * s + 2] = f4(p2, __uint_as_float(prim_shift + t));
    slot[s] = tri_shift + t;
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

// one half of a pair record (traverse.cuh, the pair-node walk): node `kid`'s box and reference (`interior_ref` when it
// is interior), `extra` in the last word.  A zero-primitive leaf owns no primitive and is never entered: its box is
// invalid and fails every slab test in the reference (Q16/Q17), enforced here with a NaN box.
__device__ __forceinline__ void pair_half(const float4* __restrict__ nodes, int64_t kid, uint32_t interior_ref, uint32_t extra,
                                          float4* q) {
    float4 a = nodes[2 * kid], b = nodes[2 * kid + 1];
    const uint32_t cm = __float_as_uint(b.w);
    const bool leaf = tr_node_leaf(cm);
    if (leaf && tr_node_count(cm) == 0u) { a.x = a.y = a.z = a.w = __int_as_float(0x7fc00000); b.x = b.y = a.x; }   // nanf("")
    const uint32_t below = (cm & TR_NODE_SPHERE_BELOW) ? TR_REF_SPHERE_BELOW : 0u;
    b.z = __uint_as_float(below | (leaf ? (TR_REF_LEAF | __float_as_uint(b.z)) : interior_ref));
    b.w = __uint_as_float(extra);
    q[0] = a;
    q[1] = b;
}

// pairs: one thread per node of the n from node0 on (pair_of: their numbering, local).  A leaf marks its last
// primitive; an interior node writes both children's halves into its pair record pair0 + pair_of, the split axis as a
// bit in the first half.
__global__ void upload_pairs(const float4* __restrict__ nodes, int64_t n, int64_t node0, uint32_t pair0,
                             const uint32_t* __restrict__ pair_of, float4* __restrict__ prims, float4* __restrict__ pairs) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t g = node0 + i;
    const float4 nb = nodes[2 * g + 1];
    const uint32_t meta = __float_as_uint(nb.w);
    if (tr_node_leaf(meta)) {
        const uint32_t cnt = tr_node_count(meta);
        if (cnt) {
            float* w = &prims[3 * (size_t)(__float_as_uint(nb.z) + cnt - 1)].w;
            *w = __uint_as_float(__float_as_uint(*w) | TR_PRIM_LAST_BIT);
        }
        return;
    }
    const int64_t kids[2] = {g + 1, (int64_t)__float_as_uint(nb.z)};
    float4* q = pairs + 4 * (size_t)(pair0 + pair_of[i]);
    for (int k = 0; k < 2; ++k)
        pair_half(nodes, kids[k], pair0 + pair_of[kids[k] - node0], k == 0 ? (1u << tr_node_axis(meta)) : 0u, q + 2 * k);
}

// an interior reference one slot up (leaf references and the sphere-below bit unchanged)
__device__ __forceinline__ void rebase_half(float4& b) {
    const uint32_t ref = __float_as_uint(b.z);
    if (!(ref & TR_REF_LEAF)) b.z = __uint_as_float(ref + 1u);
}

// the first attach after an upload: the base's nodes, pairs and shadow pairs one slot up, into new buffers, with every
// interior offset and pair reference + 1
__global__ void attach_move_base(const float4* __restrict__ nodes, int64_t n_nodes, const float4* __restrict__ pairs,
                                 int64_t n_pairs, const float4* __restrict__ shadow, int64_t n_shadow,
                                 float4* __restrict__ nodes_out, float4* __restrict__ pairs_out, float4* __restrict__ shadow_out) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n_nodes) {
        float4 b = nodes[2 * i + 1];
        if (!tr_node_leaf(__float_as_uint(b.w))) b.z = __uint_as_float(__float_as_uint(b.z) + 1u);
        nodes_out[2 * (i + 1)] = nodes[2 * i];
        nodes_out[2 * (i + 1) + 1] = b;
    }
    const float4* in[2] = {pairs, shadow};
    float4* out[2] = {pairs_out, shadow_out};
    const int64_t cnt[2] = {n_pairs, n_shadow};
    for (int t = 0; t < 2; ++t) {
        if (i >= cnt[t]) continue;
        const float4* q = in[t] + 4 * i;
        float4 h0 = q[1], h1 = q[3];
        rebase_half(h0);
        rebase_half(h1);
        float4* o = out[t] + 4 * (i + 1);
        o[0] = q[0]; o[1] = h0; o[2] = q[2]; o[3] = h1;
    }
}

// a shadow tree part's root box: the union of its pair's halves, or the vertex box of its single primitive
__device__ void shadow_root_box(const float4* __restrict__ shadow, const float4* __restrict__ prims, bool single, int64_t at,
                                float lo[3], float hi[3]) {
    for (int c = 0; c < 3; ++c) { lo[c] = TR_INF; hi[c] = -TR_INF; }
    if (single) { tri_box(xyz(prims[3 * at]), xyz(prims[3 * at + 1]), xyz(prims[3 * at + 2]), lo, hi); return; }
    for (int k = 0; k < 2; ++k) {
        const float4 a = shadow[4 * at + 2 * k], b = shadow[4 * at + 2 * k + 1];
        lo[0] = jl_min(lo[0], a.x); lo[1] = jl_min(lo[1], a.y); lo[2] = jl_min(lo[2], a.z);
        hi[0] = jl_max(hi[0], a.w); hi[1] = jl_max(hi[1], b.x); hi[2] = jl_max(hi[2], b.y);
    }
}

// node 0, pair 0 and (with_shadow) shadow pair 0 of a composed scene: base root = node 1, mesh root = node 1 + nb.  The
// split axis maximises (mesh.min + mesh.max) - (base.min + base.max) in float32, ties to the lowest axis, non-finite
// values lose, so the base is the near child when the mesh lies above it along some axis.
__global__ void attach_root(float4* nodes, float4* pairs, float4* shadow, const float4* __restrict__ prims, int64_t nb,
                            int64_t qb, int64_t pb, int64_t n_mesh, int with_shadow) {
    const float4 ba = nodes[2], bb = nodes[3], ma = nodes[2 * (1 + nb)], mb = nodes[2 * (1 + nb) + 1];
    const float blo[3] = {ba.x, ba.y, ba.z}, bhi[3] = {ba.w, bb.x, bb.y}, mlo[3] = {ma.x, ma.y, ma.z}, mhi[3] = {ma.w, mb.x, mb.y};
    uint32_t axis = 0;
    float best = 0.0f;
    bool found = false;
    float lo[3], hi[3];
    for (int k = 0; k < 3; ++k) {
        const float v = __fsub_rn(__fadd_rn(mlo[k], mhi[k]), __fadd_rn(blo[k], bhi[k]));
        if (isfinite(v) && (!found || v > best)) { best = v; axis = k; found = true; }
        lo[k] = jl_min(blo[k], mlo[k]);
        hi[k] = jl_max(bhi[k], mhi[k]);
    }
    const uint32_t meta = (axis << 30) | (__float_as_uint(bb.w) & TR_NODE_SPHERE_BELOW);
    nodes[0] = make_float4(lo[0], lo[1], lo[2], hi[0]);
    nodes[1] = make_float4(hi[1], hi[2], __uint_as_float((uint32_t)(1 + nb)), __uint_as_float(meta));
    pair_half(nodes, 1, 1u, 1u << axis, pairs);
    pair_half(nodes, 1 + nb, (uint32_t)(1 + qb), 0u, pairs + 2);
    if (!with_shadow) return;
    const int64_t at[2] = {pb == 1 ? 0 : 1, pb};
    const bool single[2] = {pb == 1, n_mesh == 1};
    for (int k = 0; k < 2; ++k) {
        shadow_root_box(shadow, prims, single[k], at[k], lo, hi);
        const uint32_t ref = single[k] ? (TR_REF_LEAF | (uint32_t)pb * k) : (uint32_t)at[k];
        shadow[2 * k] = make_float4(lo[0], lo[1], lo[2], hi[0]);
        shadow[2 * k + 1] = make_float4(hi[1], hi[2], __uint_as_float(ref), __uint_as_float(k == 0 ? 1u << axis : 0u));
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
                                                      static_cast<const uint32_t*>(d->tri_materials), order, n, 0u, 0u, 0u,
                                                      c->b_prims.as<float4>(), c->b_tnorm.as<float4>(),
                                                      c->refit.slot_tri_dev.as<uint32_t>());
        TR_CUDA(c, cudaGetLastError());
        ph.mark(s, "scatter");
        if (ctx_pack_pairs(c, n_nodes, scratch + o_pairs, scan_bytes)) return 1;
        ph.mark(s, "pairs");
    }
    if (ctx_put(c, c->b_spheres, nullptr, 0) || ctx_put(c, c->b_materials, mats.data(), mats.size() * sizeof(DeviceMaterial)) ||
        ctx_put(c, c->b_lights, lights.data(), lights.size() * sizeof(DeviceLight)))
        return 1;
    float4 root[2] = {};
    if (n_nodes > 0) TR_CUDA(c, cudaMemcpyAsync(root, c->b_nodes.p, sizeof(root), cudaMemcpyDeviceToHost, s));
    TR_CUDA(c, cudaStreamSynchronize(s));                  // (the materials / lights staging vectors move on)
    ph.mark(s, "readback");
    std::vector<uint32_t>().swap(c->refit.tri_index);
    c->refit.slot_tri_on_device = true;
    if (ctx_commit_scene(c, n_nodes, n, 0, mats, lights, n, n_nodes > 0 ? (n_nodes - 1) / 2 : 0, root, c->b_build.p))
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

// trace_scene_attach_mesh_device: the base (c->base) composed with the mesh under a new root.  Every refusal comes
// before the first write outside the build scratch, so a refused mesh leaves the previous scene as it was.
int attach(trace_ctx* c, const trace_mesh_device_desc* d, int64_t* n_nodes_out) {
    auto& B = c->base;
    const int64_t n = d->n_tris;
    if (!c->have_scene) return c->fail("mesh attach: no scene uploaded");
    if (B.n_prims == 0) return c->fail("mesh attach: the uploaded scene has no primitive");
    if (n < 1 || n >= (1ll << 30)) return c->fail("mesh attach: n_tris must be in [1, 2^30)");
    if (!d->tri_vertices) return c->fail("mesh attach: null vertex array");
    const int64_t nb = B.n_nodes, qb = B.n_pairs, pb = B.n_prims, n_prims = pb + n;
    if (n_prims >= (1ll << 30)) return c->fail("mesh attach: too many primitives (%lld in the base, %lld in the mesh)", (long long)pb, (long long)n);
    std::vector<DeviceMaterial> mats;
    std::vector<DeviceLight> lights;
    if (ctx_pack_materials(c, d->n_materials, d->materials, mats) || ctx_pack_lights(c, d->n_lights, d->lights, lights)) return 1;
    mats.insert(mats.begin(), B.materials.begin(), B.materials.end());
    lights.insert(lights.begin(), B.lights.begin(), B.lights.end());
    const int m = d->max_node_primitives < 1 ? 1 : (d->max_node_primitives < 255 ? d->max_node_primitives : 255);
    PhaseTimer ph;
    ph.on = getenv("TRACE_BVH_PROFILE") != nullptr;
    const auto t0 = std::chrono::steady_clock::now();
    if (ctx_drain(c)) return 1;
    cudaStream_t s = c->stream;
    ph.mark(s, nullptr);
    const float* v = static_cast<const float*>(d->tri_vertices);
    const float* nrm = static_cast<const float*>(d->tri_normals);
    // scratch as the upload's: the LBVH build (reused by the mesh's shadow tree), then the pair numbering
    const int64_t nn = 2 * n - 1;
    const size_t scan_bytes = pair_scan_bytes(nn, s), lbvh_bytes = lbvh_scratch_bytes(n, s);
    if (!scan_bytes || !lbvh_bytes) return c->fail("mesh attach: cannot size the sort or the scan");
    Carve k;
    k.take(lbvh_bytes);
    const size_t o_pairs = k.take(pair_scratch_bytes(nn, scan_bytes));
    TR_CUDA(c, c->b_build.ensure(k.used));
    char* scratch = c->b_build.as<char>();
    const uint32_t* order = nullptr;
    int64_t n_mesh = 0;
    switch (lbvh_mesh_build(s, v, nrm, static_cast<const uint32_t*>(d->tri_materials), d->n_materials, n, m, scratch, ph,
                            &n_mesh, &order)) {
        case LBVH_OK: break;
        case LBVH_NAN_BOUND: return c->fail("mesh attach: NaN in a triangle vertex (the scene is unchanged)");
        case LBVH_TOO_DEEP: return c->fail("mesh attach: the tree is deeper than 64 levels, the traversal stack (the scene is unchanged)");
        case LBVH_NAN_NORMAL: return c->fail("mesh attach: NaN in a triangle normal (the scene is unchanged)");
        case LBVH_BAD_MATERIAL: return c->fail("mesh attach: a material index is out of range (%lld materials; the scene is unchanged)", (long long)d->n_materials);
        default: return c->fail("mesh attach: CUDA error in the tree build (%s)", cudaGetErrorString(cudaGetLastError()));
    }
    const int64_t qm = (n_mesh - 1) / 2, n_nodes = 1 + nb + n_mesh, n_pairs = 1 + qb + qm;
    if (n_pairs > TR_REF_INDEX_MASK) return c->fail("mesh attach: too many interior nodes (the scene is unchanged)");
    // --- accepted: from here on the scene buffers are rewritten (the base's part only by the first attach's move)
    const size_t NODE = 2 * sizeof(float4), PAIR = 4 * sizeof(float4), PRIM = 3 * sizeof(float4);
    const int64_t base_shadow_pairs = B.shadow_depth > 1 ? pb - 1 : 0;
    const bool want_shadow = c->shadow_tree && B.n_spheres == 0 && B.shadow_depth > 0;
    const size_t shadow_bytes = want_shadow ? (size_t)(n_prims - 1) * PAIR : 0;
    const int T = 256;
    if (!B.moved) {
        DevBuf nodes2, pairs2, shadow2;
        TR_CUDA(c, nodes2.ensure((size_t)n_nodes * NODE));
        TR_CUDA(c, pairs2.ensure((size_t)n_pairs * PAIR));
        TR_CUDA(c, shadow2.ensure(std::max(shadow_bytes, (size_t)(base_shadow_pairs + 1) * PAIR)));
        const int64_t most = std::max(nb, std::max(qb, base_shadow_pairs));
        attach_move_base<<<blocks_for(most, T), T, 0, s>>>(c->b_nodes.as<float4>(), nb, c->b_pairs.as<float4>(), qb,
                                                          c->b_shadow.as<float4>(), base_shadow_pairs, nodes2.as<float4>(),
                                                          pairs2.as<float4>(), shadow2.as<float4>());
        TR_CUDA(c, cudaGetLastError());
        // the slot -> triangle map of a host-uploaded base goes to the device, where the mesh's part joins it
        if (!c->refit.slot_tri_on_device) {
            TR_CUDA(c, c->refit.slot_tri_dev.ensure((size_t)n_prims * 4));
            TR_CUDA(c, cudaMemcpyAsync(c->refit.slot_tri_dev.p, c->refit.tri_index.data(), (size_t)pb * 4, cudaMemcpyHostToDevice, s));
        }
        TR_CUDA(c, cudaStreamSynchronize(s));
        std::swap(c->b_nodes, nodes2);
        std::swap(c->b_pairs, pairs2);
        std::swap(c->b_shadow, shadow2);
        nodes2.release(); pairs2.release(); shadow2.release();
        std::vector<uint32_t>().swap(c->refit.tri_index);
        c->refit.slot_tri_on_device = true;
        B.moved = true;
        ph.mark(s, "move");
    }
    TR_CUDA(c, c->b_nodes.ensure_keep((size_t)n_nodes * NODE, (size_t)(1 + nb) * NODE, s));
    TR_CUDA(c, c->b_pairs.ensure_keep((size_t)n_pairs * PAIR, (size_t)(1 + qb) * PAIR, s));
    TR_CUDA(c, c->b_prims.ensure_keep((size_t)n_prims * PRIM, (size_t)pb * PRIM, s));
    TR_CUDA(c, c->b_tnorm.ensure_keep((size_t)n_prims * PRIM, (size_t)pb * PRIM, s));
    TR_CUDA(c, c->refit.slot_tri_dev.ensure_keep((size_t)n_prims * 4, (size_t)pb * 4, s));
    if (want_shadow) TR_CUDA(c, c->b_shadow.ensure_keep(shadow_bytes, (size_t)(base_shadow_pairs + 1) * PAIR, s));
    float4* nodes = c->b_nodes.as<float4>();
    if (lbvh_mesh_emit(s, n, m, scratch, nodes + 2 * (1 + nb), (uint32_t)(1 + nb), (uint32_t)pb)) return c->fail("mesh attach: CUDA error in emit");
    ph.mark(s, "emit");
    upload_scatter<<<blocks_for(n, T), T, 0, s>>>(v, nrm, static_cast<const uint8_t*>(d->tri_flags),
                                                  static_cast<const uint32_t*>(d->tri_materials), order, n, (uint32_t)B.n_tris,
                                                  (uint32_t)B.materials.size(), (uint32_t)pb, c->b_prims.as<float4>() + 3 * pb,
                                                  c->b_tnorm.as<float4>() + 3 * pb, c->refit.slot_tri_dev.as<uint32_t>() + pb);
    TR_CUDA(c, cudaGetLastError());
    ph.mark(s, "scatter");
    if (ctx_pack_pairs(c, n_mesh, scratch + o_pairs, scan_bytes, 1 + nb, 1 + qb)) return 1;
    ph.mark(s, "pairs");
    // the mesh's shadow tree after the base's pairs (its pairs and slots both start at pb), then pair 0 over the two
    int mesh_depth = 1;
    bool shadow = want_shadow;
    if (shadow && n >= 2) {
        const int rc = shadow_tree_build(s, c->b_prims.as<float4>() + 3 * pb, n, c->b_shadow.as<float4>() + 4 * pb, scratch,
                                         &mesh_depth, (uint32_t)pb);
        if (rc == LBVH_TOO_DEEP) shadow = false;
        else if (rc != LBVH_OK) return c->fail("mesh attach: shadow tree build failed (CUDA error)");
    }
    shadow = shadow && 1 + std::max(B.shadow_depth, mesh_depth) <= TR_STACK_SIZE;
    attach_root<<<1, 1, 0, s>>>(nodes, c->b_pairs.as<float4>(), c->b_shadow.as<float4>(), c->b_prims.as<float4>(), nb, qb, pb,
                                n, shadow ? 1 : 0);
    TR_CUDA(c, cudaGetLastError());
    ph.mark(s, "shadow-tree");
    if (ctx_put(c, c->b_materials, mats.data(), mats.size() * sizeof(DeviceMaterial)) ||
        ctx_put(c, c->b_lights, lights.data(), lights.size() * sizeof(DeviceLight)))
        return 1;
    float4 root[2];
    TR_CUDA(c, cudaMemcpyAsync(root, nodes, sizeof(root), cudaMemcpyDeviceToHost, s));
    TR_CUDA(c, cudaStreamSynchronize(s));
    ph.mark(s, "readback");
    ctx_publish_scene(c, n_nodes, n_prims, B.n_spheres, (int64_t)mats.size(), (int64_t)lights.size(), B.n_tris + n, n_pairs,
                      root, shadow);
    if (n_nodes_out) *n_nodes_out = n_nodes;
    if (ph.on) {
        cudaEventSynchronize(ph.ev[ph.n - 1]);
        char head[200];
        snprintf(head, sizeof(head), "scene attach mesh device: %lld triangles, %lld nodes on a base of %lld nodes", (long long)n,
                 (long long)n_mesh, (long long)nb);
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

// The pair records of the n_nodes >= 1 preorder node records from node0 on in b_nodes (a whole tree) into b_pairs from
// pair0 on (sized for them), and the last-of-leaf bit of every leaf's last primitive into b_prims; `scratch`:
// pair_scratch_bytes(n_nodes, scan_bytes) bytes
int ctx_pack_pairs(trace_ctx* c, int64_t n_nodes, char* scratch, size_t scan_bytes, int64_t node0, int64_t pair0) {
    Carve k;
    uint32_t* flag = reinterpret_cast<uint32_t*>(scratch + k.take(n_nodes * 4));
    uint32_t* pair_of = reinterpret_cast<uint32_t*>(scratch + k.take(n_nodes * 4));
    char* scan = scratch + k.take(scan_bytes);
    const float4* nodes = c->b_nodes.as<float4>();
    TR_CUDA(c, pair_numbering(c->stream, nodes + 2 * node0, n_nodes, flag, pair_of, scan, scan_bytes));
    upload_pairs<<<blocks_for(n_nodes, 256), 256, 0, c->stream>>>(nodes, n_nodes, node0, (uint32_t)pair0, pair_of,
                                                                  c->b_prims.as<float4>(), c->b_pairs.as<float4>());
    TR_CUDA(c, cudaGetLastError());
    return 0;
}

extern "C" int trace_scene_upload_mesh_device(trace_ctx* c, const trace_mesh_device_desc* d, int64_t* n_nodes_out) {
    if (!c || !d) return 1;
    cudaSetDevice(c->device);
    return upload(c, d, n_nodes_out);
}

extern "C" int trace_scene_attach_mesh_device(trace_ctx* c, const trace_mesh_device_desc* d, int64_t* n_nodes_out) {
    if (!c || !d) return 1;
    cudaSetDevice(c->device);
    return attach(c, d, n_nodes_out);
}
