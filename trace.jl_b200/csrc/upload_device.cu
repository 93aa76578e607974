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
// trace_scene_attach_meshes_device composes k such meshes with the scene of the last upload (the base) under a top
// tree, C(base, G(0, k)) of the header: every new mesh is built into its own part of the build scratch (so a refusal
// comes before any write), then written where the layout puts it by the same steps with their shifts; a kept mesh
// whose place or shifts changed goes out to the staging and back with its references rebased (place_part); then the
// top tree's nodes, pairs and shadow pairs over the parts' current root boxes (group_records).  The first attach after
// an upload moves the base's records up one slot (place_part too); later ones leave the base alone.
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

// One part of a composed scene (the base or an attached mesh) and where its records go: nodes, pair records, primitive
// and normal records, shadow pairs and the slot -> triangle map, each from its source to its destination (a count of 0
// skips that kind).  Each kind of reference has its own shift, added modulo 2^32 so that a part moving down works too.
struct PartMove {
    const float4 *nodes, *pairs, *prims, *tnorm, *shadow;
    const uint32_t* slot;
    float4 *nodes_out, *pairs_out, *prims_out, *tnorm_out, *shadow_out;
    uint32_t* slot_out;
    int64_t n_nodes, n_pairs, n_prims, n_shadow;
    uint32_t d_node, d_pair, d_prim, d_shadow, d_tri, d_mat;
};

// a child reference of a pair record: a leaf's first primitive slot + d_leaf, a pair index + d_pair (flag bits kept)
__device__ __forceinline__ void rebase_half(float4& b, uint32_t d_pair, uint32_t d_leaf) {
    const uint32_t ref = __float_as_uint(b.z);
    b.z = __uint_as_float(ref + ((ref & TR_REF_LEAF) ? d_leaf : d_pair));
}

// place / rebase: one thread per record index.  Interior offsets + d_node, leaf offsets + d_prim, pair references +
// d_pair (shadow pairs: + d_shadow), leaf references + d_prim, materials + d_mat, `original` + d_prim, slot map + d_tri.
// The first attach after an upload moves the base with d_node = d_pair = d_shadow = 1 and no primitive.
__global__ void place_part(const PartMove p) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < p.n_nodes) {
        float4 b = p.nodes[2 * i + 1];
        b.z = __uint_as_float(__float_as_uint(b.z) + (tr_node_leaf(__float_as_uint(b.w)) ? p.d_prim : p.d_node));
        p.nodes_out[2 * i] = p.nodes[2 * i];
        p.nodes_out[2 * i + 1] = b;
    }
    const float4* in[2] = {p.pairs, p.shadow};
    float4* out[2] = {p.pairs_out, p.shadow_out};
    const int64_t cnt[2] = {p.n_pairs, p.n_shadow};
    const uint32_t d_pair[2] = {p.d_pair, p.d_shadow};
    for (int t = 0; t < 2; ++t) {
        if (i >= cnt[t]) continue;
        const float4* q = in[t] + 4 * i;
        float4 h0 = q[1], h1 = q[3];
        rebase_half(h0, d_pair[t], p.d_prim);
        rebase_half(h1, d_pair[t], p.d_prim);
        float4* o = out[t] + 4 * i;
        o[0] = q[0]; o[1] = h0; o[2] = q[2]; o[3] = h1;
    }
    if (i < p.n_prims) {
        const float4* q = p.prims + 3 * i;
        float4 m = q[1], g = q[2];
        m.w = __uint_as_float(__float_as_uint(m.w) + p.d_mat);
        g.w = __uint_as_float(__float_as_uint(g.w) + p.d_prim);
        float4* o = p.prims_out + 3 * i;
        o[0] = q[0]; o[1] = m; o[2] = g;
        for (int k = 0; k < 3; ++k) p.tnorm_out[3 * i + k] = p.tnorm[3 * i + k];
        p.slot_out[i] = p.slot[i] + p.d_tri;
    }
}

int launch_place(trace_ctx* c, const PartMove& p) {
    const int64_t most = std::max(std::max(p.n_nodes, p.n_pairs), std::max(p.n_prims, p.n_shadow));
    if (most == 0) return 0;
    place_part<<<blocks_for(most, 256), 256, 0, c->stream>>>(p);
    TR_CUDA(c, cudaGetLastError());
    return 0;
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

const int MAX_MESHES = 64;

// An interior node of the top tree C(base, G(0, k)): its node, pair and shadow pair, and of each child the root node,
// its pair (when interior) and its shadow reference (a shadow pair, or TR_REF_LEAF | the slot of a single primitive)
struct GroupNode {
    uint32_t node, pair, shadow;
    uint32_t kid_node[2], kid_pair[2], kid_shadow[2];
};
struct GroupList {
    int n, with_shadow;
    GroupNode g[MAX_MESHES];      // the k - 1 nodes of G bottom-up, then node 0
};

// group records: each node of the list from its children's current root boxes, in order (children first).  The split
// axis maximises (second.min + second.max) - (first.min + first.max) in float32, ties to the lowest axis, non-finite
// values lose; the box is the Julia min / max union.  With with_shadow, its shadow pair holds the two children's shadow
// root boxes and references with the same axis bit.
__global__ void group_records(float4* nodes, float4* pairs, float4* shadow, const float4* __restrict__ prims,
                              const GroupList gl) {
    for (int i = 0; i < gl.n; ++i) {
        const GroupNode& g = gl.g[i];
        const float4 aa = nodes[2 * g.kid_node[0]], ab = nodes[2 * g.kid_node[0] + 1];
        const float4 ba = nodes[2 * g.kid_node[1]], bb = nodes[2 * g.kid_node[1] + 1];
        const float alo[3] = {aa.x, aa.y, aa.z}, ahi[3] = {aa.w, ab.x, ab.y}, blo[3] = {ba.x, ba.y, ba.z}, bhi[3] = {ba.w, bb.x, bb.y};
        uint32_t axis = 0;
        float best = 0.0f;
        bool found = false;
        float lo[3], hi[3];
        for (int k = 0; k < 3; ++k) {
            const float v = __fsub_rn(__fadd_rn(blo[k], bhi[k]), __fadd_rn(alo[k], ahi[k]));
            if (isfinite(v) && (!found || v > best)) { best = v; axis = k; found = true; }
            lo[k] = jl_min(alo[k], blo[k]);
            hi[k] = jl_max(ahi[k], bhi[k]);
        }
        const uint32_t meta = (axis << 30) | ((__float_as_uint(ab.w) | __float_as_uint(bb.w)) & TR_NODE_SPHERE_BELOW);
        nodes[2 * g.node] = make_float4(lo[0], lo[1], lo[2], hi[0]);
        nodes[2 * g.node + 1] = make_float4(hi[1], hi[2], __uint_as_float(g.kid_node[1]), __uint_as_float(meta));
        float4* q = pairs + 4 * (size_t)g.pair;
        pair_half(nodes, g.kid_node[0], g.kid_pair[0], 1u << axis, q);
        pair_half(nodes, g.kid_node[1], g.kid_pair[1], 0u, q + 2);
        if (!gl.with_shadow) continue;
        float4* sh = shadow + 4 * (size_t)g.shadow;
        for (int k = 0; k < 2; ++k) {
            const uint32_t ref = g.kid_shadow[k];
            shadow_root_box(shadow, prims, (ref & TR_REF_LEAF) != 0u, ref & TR_REF_INDEX_MASK, lo, hi);
            sh[2 * k] = make_float4(lo[0], lo[1], lo[2], hi[0]);
            sh[2 * k + 1] = make_float4(hi[1], hi[2], __uint_as_float(ref), __uint_as_float(k == 0 ? 1u << axis : 0u));
        }
    }
}

// Where G(lo, hi) of the slots puts its records when its root is node N, pair Q, primitive slot P and shadow pair S:
// each slot's position, and G's interior nodes appended to `out` bottom-up.  Returns G's sizes and root references.
struct PartInfo {
    int64_t nodes, pairs, prims;
    uint32_t root_node, root_pair, root_shadow;
};
PartInfo place_group(std::vector<trace_ctx::Slot>& sl, int lo, int hi, int64_t N, int64_t Q, int64_t P, int64_t S,
                     std::vector<GroupNode>& out) {
    if (hi - lo == 1) {
        auto& m = sl[lo];
        m.node = N; m.pair = Q; m.prim = P; m.shadow = S;
        return {m.n_nodes, m.n_pairs, m.n_tris, (uint32_t)N, (uint32_t)Q, m.n_tris == 1 ? TR_REF_LEAF | (uint32_t)P : (uint32_t)S};
    }
    const int mid = lo + (hi - lo + 1) / 2;
    const PartInfo a = place_group(sl, lo, mid, N + 1, Q + 1, P, S + 1, out);
    const PartInfo b = place_group(sl, mid, hi, N + 1 + a.nodes, Q + 1 + a.pairs, P + a.prims, S + a.prims, out);
    out.push_back({(uint32_t)N, (uint32_t)Q, (uint32_t)S, {a.root_node, b.root_node}, {a.root_pair, b.root_pair},
                   {a.root_shadow, b.root_shadow}});
    return {1 + a.nodes + b.nodes, 1 + a.pairs + b.pairs, a.prims + b.prims, (uint32_t)N, (uint32_t)Q, (uint32_t)S};
}

// the levels of G(lo, hi)'s composed shadow tree, 0 when a slot has none
int group_depth(const std::vector<trace_ctx::Slot>& sl, int lo, int hi) {
    if (hi - lo == 1) return sl[lo].shadow_depth;
    const int mid = lo + (hi - lo + 1) / 2, a = group_depth(sl, lo, mid), b = group_depth(sl, mid, hi);
    return a && b ? 1 + std::max(a, b) : 0;
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

// trace_scene_attach_meshes_device: the base (c->base) composed with k meshes, slot j built from d[j] or (NULL) kept.
// Every new mesh is built in its own part of the build scratch, and every refusal comes before the first write outside
// it, so a refused call leaves the previous scene and every slot as they were.
int attach(trace_ctx* c, int64_t k, const trace_mesh_device_desc* const* d, int64_t* n_nodes_out) {
    auto& B = c->base;
    if (!c->have_scene) return c->fail("mesh attach: no scene uploaded");
    if (B.n_prims == 0) return c->fail("mesh attach: the uploaded scene has no primitive");
    if (k < 1 || k > MAX_MESHES) return c->fail("mesh attach: n_meshes must be in [1, %d], got %lld", MAX_MESHES, (long long)k);
    if (!d) return c->fail("mesh attach: null mesh array");
    int levels = 0;                                        // ceil(log2 k): the top tree's levels above a mesh
    while ((1ll << levels) < k) ++levels;
    const int max_depth = TR_STACK_SIZE - levels;
    std::vector<trace_ctx::Slot> sl((size_t)k);
    std::vector<int> fresh, m((size_t)k, 1);
    const int64_t nb = B.n_nodes, qb = B.n_pairs, pb = B.n_prims;
    int64_t n_prims = pb;
    for (int64_t j = 0; j < k; ++j) {
        if (!d[j]) {
            if (j >= (int64_t)c->slots.size())
                return c->fail("mesh attach: mesh %lld is NULL (keep) but slot %lld holds no mesh", (long long)j, (long long)j);
            sl[j] = c->slots[j];
            if (sl[j].node_depth > max_depth)
                return c->fail("mesh attach: the tree of mesh %lld (kept) is deeper than %d levels, the traversal stack under a top tree of %lld meshes (the scene is unchanged)",
                               (long long)j, max_depth, (long long)k);
        } else {
            const int64_t n = d[j]->n_tris;
            if (n < 1 || n >= (1ll << 30)) return c->fail("mesh attach: n_tris must be in [1, 2^30) (mesh %lld)", (long long)j);
            if (!d[j]->tri_vertices) return c->fail("mesh attach: null vertex array (mesh %lld)", (long long)j);
            if (ctx_pack_materials(c, d[j]->n_materials, d[j]->materials, sl[j].materials) ||
                ctx_pack_lights(c, d[j]->n_lights, d[j]->lights, sl[j].lights))
                return 1;
            sl[j].n_tris = n;
            const int mp = d[j]->max_node_primitives;
            m[j] = mp < 1 ? 1 : (mp < 255 ? mp : 255);
            fresh.push_back((int)j);
        }
        n_prims += sl[j].n_tris;
    }
    if (n_prims >= (1ll << 30)) return c->fail("mesh attach: too many primitives (%lld in the composed scene)", (long long)n_prims);
    PhaseTimer ph, quiet;
    ph.on = getenv("TRACE_BVH_PROFILE") != nullptr;
    const auto t0 = std::chrono::steady_clock::now();
    if (ctx_drain(c)) return 1;
    cudaStream_t s = c->stream;
    ph.mark(s, nullptr);
    // scratch: each new mesh's LBVH build (reused by its shadow tree), the pair numbering's, the builds' status blocks,
    // then the staging of the kept meshes that move (sized once the layout is known)
    Carve kv;
    std::vector<size_t> o_lbvh((size_t)k), o_order((size_t)k), o_stage((size_t)k);
    int64_t most = 1;
    for (int j : fresh) {
        const size_t bytes = lbvh_scratch_bytes(sl[j].n_tris, s);
        if (!bytes) return c->fail("mesh attach: cannot size the sort");
        o_lbvh[j] = kv.take(bytes);
        most = std::max(most, 2 * sl[j].n_tris - 1);
    }
    const size_t scan_bytes = pair_scan_bytes(most, s);
    if (!scan_bytes) return c->fail("mesh attach: cannot size the scan");
    const size_t SB = lbvh_status_bytes();
    const size_t o_pairs = kv.take(pair_scratch_bytes(most, scan_bytes)), o_status = kv.take(std::max<size_t>(1, fresh.size()) * SB);
    const size_t build_used = kv.used;
    TR_CUDA(c, c->b_build.ensure(build_used));
    // every build enqueued, their status blocks gathered and read back once
    std::vector<char> status(std::max<size_t>(1, fresh.size()) * SB);
    auto read_status = [&](const std::vector<int>& which, auto scratch_of) -> int {
        char* scratch = c->b_build.as<char>();
        for (size_t i = 0; i < which.size(); ++i)
            TR_CUDA(c, cudaMemcpyAsync(scratch + o_status + i * SB, lbvh_status(scratch_of(which[i]), sl[which[i]].n_tris), SB,
                                       cudaMemcpyDeviceToDevice, s));
        if (which.empty()) return 0;
        TR_CUDA(c, cudaMemcpyAsync(status.data(), scratch + o_status, which.size() * SB, cudaMemcpyDeviceToHost, s));
        TR_CUDA(c, cudaStreamSynchronize(s));
        return 0;
    };
    for (int j : fresh) {
        const trace_mesh_device_desc* dj = d[j];
        if (lbvh_mesh_enqueue(s, static_cast<const float*>(dj->tri_vertices), static_cast<const float*>(dj->tri_normals),
                              static_cast<const uint32_t*>(dj->tri_materials), dj->n_materials, sl[j].n_tris, m[j],
                              c->b_build.as<char>() + o_lbvh[j], quiet))
            return c->fail("mesh attach: CUDA error in the tree build (%s)", cudaGetErrorString(cudaGetLastError()));
    }
    if (read_status(fresh, [&](int j) { return c->b_build.as<char>() + o_lbvh[j]; })) return 1;
    for (size_t i = 0; i < fresh.size(); ++i) {
        const int j = fresh[i];
        const trace_mesh_device_desc* dj = d[j];
        char* scratch = c->b_build.as<char>();
        const uint32_t* order = nullptr;
        int depth = 0;
        switch (lbvh_mesh_result(status.data() + i * SB, scratch + o_lbvh[j], sl[j].n_tris, &sl[j].n_nodes, &order, &depth)) {
            case LBVH_OK: break;
            case LBVH_NAN_BOUND: return c->fail("mesh attach: NaN in a triangle vertex (mesh %d; the scene is unchanged)", j);
            case LBVH_TOO_DEEP: return c->fail("mesh attach: the tree is deeper than 64 levels, the traversal stack (mesh %d; the scene is unchanged)", j);
            case LBVH_NAN_NORMAL: return c->fail("mesh attach: NaN in a triangle normal (mesh %d; the scene is unchanged)", j);
            case LBVH_BAD_MATERIAL: return c->fail("mesh attach: a material index is out of range (mesh %d, %lld materials; the scene is unchanged)", j, (long long)dj->n_materials);
            default: return c->fail("mesh attach: CUDA error in the tree build (%s)", cudaGetErrorString(cudaGetLastError()));
        }
        if (depth > max_depth)
            return c->fail("mesh attach: the tree of mesh %d is deeper than %d levels, the traversal stack under a top tree of %lld meshes (the scene is unchanged)",
                           j, max_depth, (long long)k);
        sl[j].n_pairs = (sl[j].n_nodes - 1) / 2;           // a full binary tree
        sl[j].node_depth = depth;
        o_order[j] = (size_t)(reinterpret_cast<const char*>(order) - scratch);
    }
    ph.mark(s, "build");
    // the layout: triangles and materials in slot order, records where C(base, G(0, k)) puts them
    int64_t tri = B.n_tris, mat = (int64_t)B.materials.size();
    for (auto& q : sl) { q.tri = tri; q.material = mat; tri += q.n_tris; mat += (int64_t)q.materials.size(); }
    std::vector<GroupNode> groups;
    const PartInfo g = place_group(sl, 0, (int)k, 1 + nb, 1 + qb, pb, pb, groups);
    groups.push_back({0u, 0u, 0u, {1u, g.root_node}, {1u, g.root_pair}, {pb == 1 ? TR_REF_LEAF : 1u, g.root_shadow}});
    const int64_t n_nodes = 1 + nb + g.nodes, n_pairs = 1 + qb + g.pairs;
    if (n_pairs > TR_REF_INDEX_MASK) return c->fail("mesh attach: too many interior nodes (the scene is unchanged)");
    const size_t NODE = 2 * sizeof(float4), PAIR = 4 * sizeof(float4), PRIM = 3 * sizeof(float4);
    const bool want_shadow = c->shadow_tree && B.n_spheres == 0 && B.shadow_depth > 0;
    std::vector<int> moved;                                // kept slots whose records or references move
    for (int64_t j = 0; j < k; ++j) {
        if (d[j]) continue;
        const auto &o = c->slots[j], &q = sl[j];
        if (o.node == q.node && o.pair == q.pair && o.prim == q.prim && o.shadow == q.shadow && o.tri == q.tri &&
            o.material == q.material)
            continue;
        moved.push_back((int)j);
        // its shadow pairs move along only when they are valid and this call keeps shadow trees; else it has none
        if (!(want_shadow && o.shadow_depth > 1)) sl[j].shadow_depth = q.n_tris == 1 ? 1 : 0;
        o_stage[j] = kv.take((size_t)q.n_nodes * NODE);
        kv.take((size_t)q.n_pairs * PAIR); kv.take((size_t)q.n_tris * PRIM); kv.take((size_t)q.n_tris * PRIM);
        kv.take(q.shadow_depth > 1 ? (size_t)(q.n_tris - 1) * PAIR : 0); kv.take((size_t)q.n_tris * 4);
    }
    // --- accepted: from here on the scene buffers are rewritten (the base's part only by the first attach's move)
    TR_CUDA(c, c->b_build.ensure_keep(kv.used, build_used, s));
    const int64_t base_shadow_pairs = B.shadow_depth > 1 ? pb - 1 : 0;
    const size_t shadow_bytes = want_shadow ? (size_t)(n_prims - 1) * PAIR : 0;
    int64_t old_nodes = c->scene.n_nodes, old_pairs = c->refit.n_pairs, old_prims = c->scene.n_prims;
    if (!B.moved) {
        DevBuf nodes2, pairs2, shadow2;
        TR_CUDA(c, nodes2.ensure((size_t)n_nodes * NODE));
        TR_CUDA(c, pairs2.ensure((size_t)n_pairs * PAIR));
        TR_CUDA(c, shadow2.ensure(std::max(shadow_bytes, (size_t)(base_shadow_pairs + 1) * PAIR)));
        PartMove mv{};
        mv.nodes = c->b_nodes.as<float4>(); mv.pairs = c->b_pairs.as<float4>(); mv.shadow = c->b_shadow.as<float4>();
        mv.nodes_out = nodes2.as<float4>() + 2; mv.pairs_out = pairs2.as<float4>() + 4; mv.shadow_out = shadow2.as<float4>() + 4;
        mv.n_nodes = nb; mv.n_pairs = qb; mv.n_shadow = base_shadow_pairs;
        mv.d_node = mv.d_pair = mv.d_shadow = 1u;
        if (launch_place(c, mv)) return 1;
        // the slot -> triangle map of a host-uploaded base goes to the device, where the meshes' parts join it
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
        old_nodes = 1 + nb; old_pairs = 1 + qb; old_prims = pb;
        ph.mark(s, "move");
    }
    const int64_t old_shadow = old_prims - 1;
    TR_CUDA(c, c->b_nodes.ensure_keep((size_t)n_nodes * NODE, std::min(c->b_nodes.bytes, (size_t)old_nodes * NODE), s));
    TR_CUDA(c, c->b_pairs.ensure_keep((size_t)n_pairs * PAIR, std::min(c->b_pairs.bytes, (size_t)old_pairs * PAIR), s));
    TR_CUDA(c, c->b_prims.ensure_keep((size_t)n_prims * PRIM, std::min(c->b_prims.bytes, (size_t)old_prims * PRIM), s));
    TR_CUDA(c, c->b_tnorm.ensure_keep((size_t)n_prims * PRIM, std::min(c->b_tnorm.bytes, (size_t)old_prims * PRIM), s));
    TR_CUDA(c, c->refit.slot_tri_dev.ensure_keep((size_t)n_prims * 4, std::min(c->refit.slot_tri_dev.bytes, (size_t)old_prims * 4), s));
    if (want_shadow) TR_CUDA(c, c->b_shadow.ensure_keep(shadow_bytes, std::min(c->b_shadow.bytes, (size_t)old_shadow * PAIR), s));
    float4 *nodes = c->b_nodes.as<float4>(), *pairs = c->b_pairs.as<float4>(), *prims = c->b_prims.as<float4>();
    float4 *tnorm = c->b_tnorm.as<float4>(), *shadow_pairs = c->b_shadow.as<float4>();
    uint32_t* slot = c->refit.slot_tri_dev.as<uint32_t>();
    char* scratch = c->b_build.as<char>();
    // the kept meshes that move: out to the staging with their new references (all read before anything is written)
    size_t kept_bytes = 0;
    std::vector<PartMove> back;
    for (int j : moved) {
        const auto &o = c->slots[j], &q = sl[j];
        Carve st;
        const size_t on = st.take((size_t)q.n_nodes * NODE), oq = st.take((size_t)q.n_pairs * PAIR),
                     op = st.take((size_t)q.n_tris * PRIM), ot = st.take((size_t)q.n_tris * PRIM),
                     os = st.take(q.shadow_depth > 1 ? (size_t)(q.n_tris - 1) * PAIR : 0), ol = st.take((size_t)q.n_tris * 4);
        char* at = scratch + o_stage[j];
        PartMove mv{};
        mv.nodes = nodes + 2 * o.node; mv.pairs = pairs + 4 * o.pair; mv.prims = prims + 3 * o.prim; mv.tnorm = tnorm + 3 * o.prim;
        mv.shadow = shadow_pairs + 4 * o.shadow; mv.slot = slot + o.prim;
        mv.nodes_out = (float4*)(at + on); mv.pairs_out = (float4*)(at + oq); mv.prims_out = (float4*)(at + op);
        mv.tnorm_out = (float4*)(at + ot); mv.shadow_out = (float4*)(at + os); mv.slot_out = (uint32_t*)(at + ol);
        mv.n_nodes = q.n_nodes; mv.n_pairs = q.n_pairs; mv.n_prims = q.n_tris; mv.n_shadow = q.shadow_depth > 1 ? q.n_tris - 1 : 0;
        mv.d_node = (uint32_t)(q.node - o.node); mv.d_pair = (uint32_t)(q.pair - o.pair); mv.d_prim = (uint32_t)(q.prim - o.prim);
        mv.d_shadow = (uint32_t)(q.shadow - o.shadow); mv.d_tri = (uint32_t)(q.tri - o.tri);
        mv.d_mat = (uint32_t)(q.material - o.material);
        if (launch_place(c, mv)) return 1;
        // ... and back into the scene at the new position, unchanged
        PartMove bk{};
        bk.nodes = mv.nodes_out; bk.pairs = mv.pairs_out; bk.prims = mv.prims_out; bk.tnorm = mv.tnorm_out;
        bk.shadow = mv.shadow_out; bk.slot = mv.slot_out;
        bk.nodes_out = nodes + 2 * q.node; bk.pairs_out = pairs + 4 * q.pair; bk.prims_out = prims + 3 * q.prim;
        bk.tnorm_out = tnorm + 3 * q.prim; bk.shadow_out = shadow_pairs + 4 * q.shadow; bk.slot_out = slot + q.prim;
        bk.n_nodes = mv.n_nodes; bk.n_pairs = mv.n_pairs; bk.n_prims = mv.n_prims; bk.n_shadow = mv.n_shadow;
        back.push_back(bk);
        kept_bytes += st.used;
    }
    ph.mark(s, "stage");
    // the new meshes at their places: the upload's emit, scatter and pair packing with their shifts
    for (int j : fresh) {
        const auto& q = sl[j];
        const trace_mesh_device_desc* dj = d[j];
        if (lbvh_mesh_emit(s, q.n_tris, m[j], scratch + o_lbvh[j], nodes + 2 * q.node, (uint32_t)q.node, (uint32_t)q.prim))
            return c->fail("mesh attach: CUDA error in emit");
        upload_scatter<<<blocks_for(q.n_tris, 256), 256, 0, s>>>(
            static_cast<const float*>(dj->tri_vertices), static_cast<const float*>(dj->tri_normals),
            static_cast<const uint8_t*>(dj->tri_flags), static_cast<const uint32_t*>(dj->tri_materials),
            reinterpret_cast<const uint32_t*>(scratch + o_order[j]), q.n_tris, (uint32_t)q.tri,
            (uint32_t)q.material, (uint32_t)q.prim, prims + 3 * q.prim, tnorm + 3 * q.prim, slot + q.prim);
        TR_CUDA(c, cudaGetLastError());
        if (ctx_pack_pairs(c, q.n_nodes, scratch + o_pairs, scan_bytes, q.node, q.pair)) return 1;
    }
    ph.mark(s, "meshes");
    for (const PartMove& bk : back) if (launch_place(c, bk)) return 1;
    ph.mark(s, "place");
    // each new mesh's shadow tree at its place (its scratch is free again; the status blocks read back once), then the
    // top tree's records
    std::vector<int> shadowed;
    for (int j : fresh) {
        auto& q = sl[j];
        q.shadow_depth = q.n_tris == 1 ? 1 : 0;
        if (!want_shadow || q.n_tris < 2) continue;
        if (shadow_tree_enqueue(s, prims + 3 * q.prim, q.n_tris, scratch + o_lbvh[j]))
            return c->fail("mesh attach: shadow tree build failed (CUDA error)");
        shadowed.push_back(j);
    }
    if (read_status(shadowed, [&](int j) { return scratch + o_lbvh[j]; })) return 1;
    for (size_t i = 0; i < shadowed.size(); ++i) {
        auto& q = sl[shadowed[i]];
        const int rc = shadow_tree_emit(s, status.data() + i * SB, q.n_tris, scratch + o_lbvh[shadowed[i]],
                                        shadow_pairs + 4 * q.shadow, &q.shadow_depth, (uint32_t)q.shadow, (uint32_t)q.prim);
        if (rc == LBVH_TOO_DEEP) q.shadow_depth = 0;
        else if (rc != LBVH_OK) return c->fail("mesh attach: shadow tree build failed (CUDA error)");
    }
    ph.mark(s, "shadow-tree");
    const int gd = group_depth(sl, 0, (int)k);
    const bool shadow = want_shadow && gd > 0 && 1 + std::max(B.shadow_depth, gd) <= TR_STACK_SIZE;
    GroupList gl;
    gl.n = (int)groups.size();
    gl.with_shadow = shadow ? 1 : 0;
    std::copy(groups.begin(), groups.end(), gl.g);
    group_records<<<1, 1, 0, s>>>(nodes, pairs, shadow_pairs, prims, gl);
    TR_CUDA(c, cudaGetLastError());
    ph.mark(s, "top");
    std::vector<DeviceMaterial> mats = B.materials;
    std::vector<DeviceLight> lights = B.lights;
    for (const auto& q : sl) {
        mats.insert(mats.end(), q.materials.begin(), q.materials.end());
        lights.insert(lights.end(), q.lights.begin(), q.lights.end());
    }
    if (ctx_put(c, c->b_materials, mats.data(), mats.size() * sizeof(DeviceMaterial)) ||
        ctx_put(c, c->b_lights, lights.data(), lights.size() * sizeof(DeviceLight)))
        return 1;
    float4 root[2];
    TR_CUDA(c, cudaMemcpyAsync(root, nodes, sizeof(root), cudaMemcpyDeviceToHost, s));
    TR_CUDA(c, cudaStreamSynchronize(s));
    ph.mark(s, "readback");
    c->slots.swap(sl);
    ctx_publish_scene(c, n_nodes, n_prims, B.n_spheres, (int64_t)mats.size(), (int64_t)lights.size(), tri, n_pairs, root,
                      shadow);
    if (n_nodes_out) *n_nodes_out = n_nodes;
    if (ph.on) {
        cudaEventSynchronize(ph.ev[ph.n - 1]);
        char head[240];
        snprintf(head, sizeof(head), "scene attach mesh device: %lld meshes, %zu built, %zu kept moved (%zu bytes staged), %lld nodes on a base of %lld nodes",
                 (long long)k, fresh.size(), moved.size(), kept_bytes, (long long)n_nodes, (long long)nb);
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

extern "C" int trace_scene_attach_meshes_device(trace_ctx* c, int64_t n_meshes, const trace_mesh_device_desc* const* meshes,
                                                int64_t* n_nodes_out) {
    if (!c) return 1;
    cudaSetDevice(c->device);
    return attach(c, n_meshes, meshes, n_nodes_out);
}

extern "C" int trace_scene_attach_mesh_device(trace_ctx* c, const trace_mesh_device_desc* d, int64_t* n_nodes_out) {
    if (!c || !d) return 1;
    cudaSetDevice(c->device);
    return attach(c, 1, &d, n_nodes_out);
}
