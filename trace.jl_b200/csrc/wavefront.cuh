// wavefront.cuh — the two traversal stages shared by the Whitted and SPPM wavefronts: `extend` (closest hit over a ray
// queue) and `shadow` (any hit over a shadow queue, fused with the accumulate: an unoccluded ray adds its
// contribution to the accumulator slot it names).  Queue sizes live in device memory, so the kernels are launched
// as persistent grid-stride grids (a multiple of the SM count) and no host round trip sits between stages.
#pragma once
#include "context.hpp"
#include "shading.cuh"

// Traversal kernels are bound by dependent-fetch latency, so resident warps matter more than registers: capping them
// at 64 registers (8 CTAs of 128 threads per SM instead of 7 at 69 registers; 20 B of spills) measured +12 % on tess-1M;
// 9 CTAs (56 registers) +9 %, 10 CTAs (48 registers, 76 B spills) +4 % (profiles/r1_experiments.md).
#ifndef TR_TRAV_MIN_BLOCKS
#define TR_TRAV_MIN_BLOCKS 8
#endif
// WAIT: 0 = plain per-thread loop (traverse<>), > 0 = warp-synchronous loop with batched leaves (traverse_lb<>).
// The grid-stride loop is warp-uniform (whole warps step together; lanes past the end of the queue are `valid ==
// false`), which the warp-synchronous traversal needs and the plain one does not mind.
// Two-ended queues (Whitted, bounce levels >= 2): a glass hit spawns a reflected AND a transmitted ray; pushed into one
// queue they alternate in blocks and every warp of the next level walks two unrelated ray bundles (ncu: 10-12 of 32
// lanes at the deep levels).  The shade stage therefore pushes reflected rays from the front (count) and transmitted
// rays from the back (count_back) of the same array: entry j < nf sits at j, entry nf + k at cap - 1 - k, so warps are
// homogeneous except the one that straddles the seam.  count_back == nullptr: a plain front-filled queue (SPPM).
__device__ __forceinline__ int queue_position(int j, int nf, int cap) { return j < nf ? j : cap - 1 - (j - nf); }
__device__ __forceinline__ void queue_extent(const int* count, const int* count_back, int cap, int& nf, int& n) {
    nf = min(*count, cap);
    n = nf + (count_back ? min(*count_back, cap - nf) : 0);
}

template <int SLAB, bool COUNT, int WAIT, bool TREE>       // TREE: walk the shadow tree (traverse_closest)
__global__ void __launch_bounds__(128, TR_TRAV_MIN_BLOCKS) k_wh_extend(DeviceScene sc, const float4* __restrict__ ro, const float4* __restrict__ rd,
                                                   const int* __restrict__ count, const int* __restrict__ count_back, int cap,
                                                   float4* __restrict__ hits, unsigned long long* counters, int* error_flag) {
    int nf, n;
    queue_extent(count, count_back, cap, nf, n);
    const int lane = threadIdx.x & 31;
    for (int base = blockIdx.x * blockDim.x + (threadIdx.x - lane); base < n; base += gridDim.x * blockDim.x) {
        const int j = base + lane;
        const bool valid = j < n;
        const int i = valid ? queue_position(j, nf, cap) : 0;
        const float4 o = valid ? q_load(&ro[i]) : make_float4(0.0f, 0.0f, 0.0f, 0.0f), d = valid ? q_load(&rd[i]) : make_float4(1.0f, 1.0f, 1.0f, 0.0f);
        HitRecord h;
        // closest hit; the third barycentric is rebuilt exactly in the shade stage from the winning triangle
        traverse_closest<SLAB, COUNT, WAIT, TREE>(sc, valid, xyz(o), xyz(d), o.w, h, counters, error_flag);
        if (valid) q_store(&hits[i], make_float4(h.t, __uint_as_float(h.prim), h.b0, h.b1));
    }
}

// TREE: walk the shadow tree (traverse_shadow; sc.shadow_pairs is set), else the reference tree
template <int SLAB, bool COUNT, int WAIT, bool TREE>
__global__ void __launch_bounds__(128, TR_TRAV_MIN_BLOCKS) k_wh_shadow(DeviceScene sc, const float4* __restrict__ so, const float4* __restrict__ sd,
                                                   const float4* __restrict__ contrib, const int* __restrict__ count, int cap,
                                                   float4* __restrict__ accum, unsigned long long* counters, int* error_flag) {
    const int n = min(*count, cap);
    const int lane = threadIdx.x & 31;
    for (int base = blockIdx.x * blockDim.x + (threadIdx.x - lane); base < n; base += gridDim.x * blockDim.x) {
        const int i = base + lane;
        const bool valid = i < n;
        const float4 o = valid ? q_load(&so[i]) : make_float4(0.0f, 0.0f, 0.0f, 0.0f), d = valid ? q_load(&sd[i]) : make_float4(1.0f, 1.0f, 1.0f, 0.0f);
        bool occ;
        if (TREE) occ = !valid || traverse_shadow<COUNT>(sc, xyz(o), xyz(d), o.w, counters, error_flag);
        else {
            HitRecord h;
            occ = traverse_any<SLAB, true, COUNT, WAIT>(sc, valid, xyz(o), xyz(d), o.w, h, counters, error_flag);
        }
        if (!occ && valid) {
            const float4 c = q_load(&contrib[i]);
            atomicAdd(&accum[__float_as_int(d.w)], make_float4(c.x, c.y, c.z, 0.0f));   // 128-bit vector atomic (sm_90+)
        }
    }
}

// exact third barycentric of the winning triangle: e2 * inv_det of the same edge functions (pure function of ray + triangle)
__device__ __forceinline__ float third_barycentric(const DeviceScene& sc, uint32_t prim, float3 o, float3 d) {
    const float4 A = __ldg(&sc.prims[3 * prim]);
    if (__float_as_uint(A.w) & TR_PRIM_SPHERE_BIT) return 0.0f;
    const float4 B = __ldg(&sc.prims[3 * prim + 1]), C = __ldg(&sc.prims[3 * prim + 2]);
    const RayPrep r = prepare_ray(o, d);
    float t, b0, b1, b2 = 0.0f;
    triangle_test(A, B, C, r, TR_INF, t, b0, b1, b2);
    return b2;
}

static void launch_extend_plain(trace_ctx* c, DeviceScene sc, const float4* ro, const float4* rd, const int* count,
                                const int* count_back, int cap, float4* hits, unsigned long long* counters, int* err) {
    c->kev_begin(0);
    trav_dispatch(c, [&](auto S, auto C_, auto W) {
        constexpr int s = decltype(S)::value, w = decltype(W)::value;
        constexpr bool cn = decltype(C_)::value;
        auto k = k_wh_extend<s, cn, w, false>;
        if constexpr (shadow_walk_capable<s, cn, w>) if (sc.shadow_pairs) k = k_wh_extend<s, cn, w, true>;
        k<<<persistent_grid(c, 16), 128, 0, c->cur_stream>>>(sc, ro, rd, count, count_back, cap, hits, counters, err);
    });
    c->stats.kernel_launches++;
    c->kev_end();
}
static void launch_shadow_plain(trace_ctx* c, DeviceScene sc, const float4* so, const float4* sd, const float4* contrib,
                                const int* count, int cap, float4* accum, unsigned long long* counters, int* err) {
    c->kev_begin(1);
    trav_dispatch(c, [&](auto S, auto C_, auto W) {
        constexpr int s = decltype(S)::value, w = decltype(W)::value;
        constexpr bool cn = decltype(C_)::value;
        auto k = k_wh_shadow<s, cn, w, false>;
        if constexpr (shadow_walk_capable<s, cn, w>) if (sc.shadow_pairs) k = k_wh_shadow<s, cn, w, true>;
        k<<<persistent_grid(c, 16), 128, 0, c->cur_stream>>>(sc, so, sd, contrib, count, cap, accum, counters, err);
    });
    c->stats.kernel_launches++;
    c->kev_end();
}

static void launch_extend(trace_ctx* c, int grid, DeviceScene sc, const float4* ro, const float4* rd, const int* count, int cap,
                          float4* hits, unsigned long long* counters, int* err, const int* count_back = nullptr) {
    launch_extend_plain(c, hit_launch_scene(c, sc), ro, rd, count, count_back, cap, hits, counters, err);
}
static void launch_shadow(trace_ctx* c, int grid, DeviceScene sc, const float4* so, const float4* sd, const float4* contrib,
                          const int* count, int cap, float4* accum, unsigned long long* counters, int* err) {
    launch_shadow_plain(c, shadow_launch_scene(c, sc), so, sd, contrib, count, cap, accum, counters, err);
}
