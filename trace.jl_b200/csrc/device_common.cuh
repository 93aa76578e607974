// device_common.cuh — float3 helpers, device scene layout and queue primitives of libtrace_cuda.so.
//
// Arithmetic policy: the library is compiled with -fmad=false and default -prec-div/-prec-sqrt, so every float
// operation below is a single IEEE-754 round-to-nearest op, exactly like the reference's Julia code (which LLVM never
// contracts into FMA, SURVEY.md §9 Q20).  Sums are written in the association order the reference's
// StaticArrays/GeometryBasics expressions generate (left to right).
#pragma once
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/trace_cuda.h"

namespace cg = cooperative_groups;

#define TR_INF __int_as_float(0x7f800000)
#define TR_PI 3.1415927f

// ------------------------------------------------------------------ float3
__host__ __device__ __forceinline__ float3 f3(float x, float y, float z) { return make_float3(x, y, z); }
__host__ __device__ __forceinline__ float3 f3s(float s) { return make_float3(s, s, s); }
__host__ __device__ __forceinline__ float3 operator+(float3 a, float3 b) { return f3(a.x + b.x, a.y + b.y, a.z + b.z); }
__host__ __device__ __forceinline__ float3 operator-(float3 a, float3 b) { return f3(a.x - b.x, a.y - b.y, a.z - b.z); }
__host__ __device__ __forceinline__ float3 operator-(float3 a) { return f3(-a.x, -a.y, -a.z); }
__host__ __device__ __forceinline__ float3 operator*(float3 a, float s) { return f3(a.x * s, a.y * s, a.z * s); }
__host__ __device__ __forceinline__ float3 operator*(float s, float3 a) { return f3(s * a.x, s * a.y, s * a.z); }
__host__ __device__ __forceinline__ float3 operator*(float3 a, float3 b) { return f3(a.x * b.x, a.y * b.y, a.z * b.z); }
__host__ __device__ __forceinline__ float3 operator/(float3 a, float s) { return f3(a.x / s, a.y / s, a.z / s); }
__host__ __device__ __forceinline__ float dot3(float3 a, float3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
__host__ __device__ __forceinline__ float3 cross3(float3 a, float3 b) {
    return f3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
__device__ __forceinline__ float length3(float3 a) { return sqrtf((a.x * a.x + a.y * a.y) + a.z * a.z); }
__device__ __forceinline__ float3 normalize3(float3 a) { float inv = 1.0f / length3(a); return f3(inv * a.x, inv * a.y, inv * a.z); }
__device__ __forceinline__ bool is_black3(float3 a) { return a.x == 0.0f && a.y == 0.0f && a.z == 0.0f; }
__device__ __forceinline__ float3 xyz(float4 v) { return f3(v.x, v.y, v.z); }
__device__ __forceinline__ float4 f4(float3 v, float w) { return make_float4(v.x, v.y, v.z, w); }
__device__ __forceinline__ float clampf(float x, float lo, float hi) { return x > hi ? hi : (x < lo ? lo : x); }
__device__ __forceinline__ float luminance(float3 c) { return (0.212671f * c.x + 0.715160f * c.y) + 0.072169f * c.z; }

// row-major 4x4 application (src/transformations.jl:132-144)
__device__ __forceinline__ float3 xform_point(const float* __restrict__ m, float3 p) {
    float x = ((m[0] * p.x + m[1] * p.y) + m[2] * p.z) + m[3] * 1.0f;
    float y = ((m[4] * p.x + m[5] * p.y) + m[6] * p.z) + m[7] * 1.0f;
    float z = ((m[8] * p.x + m[9] * p.y) + m[10] * p.z) + m[11] * 1.0f;
    float w = ((m[12] * p.x + m[13] * p.y) + m[14] * p.z) + m[15] * 1.0f;
    if (w == 1.0f) return f3(x, y, z);
    return f3(x / w, y / w, z / w);
}
__device__ __forceinline__ float3 xform_vector(const float* __restrict__ m, float3 v) {
    return f3((m[0] * v.x + m[1] * v.y) + m[2] * v.z, (m[4] * v.x + m[5] * v.y) + m[6] * v.z,
              (m[8] * v.x + m[9] * v.y) + m[10] * v.z);
}
__device__ __forceinline__ float3 xform_normal(const float* __restrict__ im, float3 n) {   // transpose(inv_m[1:3,1:3]) * n
    return f3((im[0] * n.x + im[4] * n.y) + im[8] * n.z, (im[1] * n.x + im[5] * n.y) + im[9] * n.z,
              (im[2] * n.x + im[6] * n.y) + im[10] * n.z);
}

// ------------------------------------------------------------------ device scene (all arrays live in HBM)
// nodes : 2 x float4 per node  {bmin.xyz, bmax.x} {bmax.y, bmax.z, offset(bits), meta(bits)}          32 B
// prims : 3 x float4 per BVH-ordered primitive                                                          48 B
//           triangle {p0.xyz, tag = 0} {p1.xyz, material} {p2.xyz, original}
//           sphere   {0,0,0,   tag = 0x80000000 | sphere index} {0,0,0, material} {0,0,0, original}
// tnorm : 3 x float4 per BVH-ordered primitive {n0.xyz, flags} {n1.xyz, 0} {n2.xyz, 0}   (read by shading only)
struct DeviceSphere {
    float m[16];
    float inv_m[16];
    float radius, z_min, z_max, theta_min, theta_max, phi_max;
    uint32_t flip, pad;
};
struct DeviceMaterial {
    uint32_t kind;
    float a[3], b[3];
    float eta;
    float alpha_u, alpha_v;      // Trowbridge-Reitz alphas, remapped + clamped on upload
    uint32_t specular;           // glass: u_roughness == 0 && v_roughness == 0
    uint32_t pad;
};
struct DeviceLight {
    uint32_t kind;
    float m[16], inv_m[16];
    float I[3], pos[3];
    float cos_total, cos_falloff;
};
struct DeviceScene {
    const float4* nodes;
    const float4* pairs;      // 4 x float4 per INTERIOR node: both children's boxes + references (traverse.cuh, pair-node walk)
    uint32_t root_ref;        // reference of the root: pair index 0, or TR_REF_LEAF | 0 when the tree is a single leaf
    const float4* prims;
    const float4* tnorm;
    const DeviceSphere* spheres;
    const DeviceMaterial* materials;
    const DeviceLight* lights;
    int n_nodes, n_prims, n_spheres, n_materials, n_lights;
    float scene_scale;        // largest |coordinate| of the root bounds (slack of the guarded slab test)
    // the shadow tree (api.cu, traverse.cuh traverse_shadow): an LBVH over the same primitive slots, one primitive per
    // leaf, n_prims - 1 pair records in the layout of `pairs`, root = pair 0.  Null: no shadow tree (analytic spheres,
    // fewer than 2 primitives, NaN vertices, deeper than 64 levels), or the launch does not use it (option shadow_tree)
    const float4* shadow_pairs;
};
struct DeviceCamera {
    float r2c[16], c2w[16];
    float lens_radius, focal_distance, shutter_open, shutter_close;
};
struct DeviceFilm {
    int crop_x0, crop_y0, crop_x1, crop_y1;
    int sb_x0, sb_y0, sb_x1, sb_y1;      // get_sample_bounds, film.jl:68-73
    int tiles_x, tiles_y;                // 16x16 sample tiles, integrators/sampler.jl:14-20
    float rx, ry, inv_rx, inv_ry;
    const float* table;                  // 16x16 [y][x] in HBM
    int width, height;
};

// ------------------------------------------------------------------ queue traffic: streamed once, evict-first
// Ray / hit / shadow queues are written by one kernel and read once by the next; the BVH (64 MB of pair nodes + 48 MB
// of primitives on tess-1M) is what should stay in the 126 MB L2.  ld.global.cs / st.global.cs mark the queue lines
// evict-first.
#ifdef TR_NO_STREAM_HINTS
__device__ __forceinline__ float4 q_load(const float4* p) { return *p; }
__device__ __forceinline__ void q_store(float4* p, float4 v) { *p = v; }
#else
__device__ __forceinline__ float4 q_load(const float4* p) { return __ldcs(p); }
__device__ __forceinline__ void q_store(float4* p, float4 v) { __stcs(p, v); }
#endif

// ------------------------------------------------------------------ queue push with warp-aggregated atomics
__device__ __forceinline__ int queue_claim(int* counter) {
    cg::coalesced_group g = cg::coalesced_threads();
    int base = 0;
    if (g.thread_rank() == 0) base = atomicAdd(counter, (int)g.size());
    base = g.shfl(base, 0);
    return base + (int)g.thread_rank();
}

// Counter-based RNG (DESIGN.md "RNG"), bit-identical to the oracle's ref::rng_uniform.
__device__ __forceinline__ float rng_uniform(uint64_t seed, uint32_t a, uint32_t b, uint32_t c) {
    uint64_t z = seed ^ ((uint64_t)a * 0x9E3779B97F4A7C15ull) ^ ((((uint64_t)b << 32) | (uint64_t)c) * 0xD1B54A32D192ED03ull);
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    return (float)(z >> 40) * 5.9604644775390625e-8f;
}
