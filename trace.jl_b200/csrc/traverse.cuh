// traverse.cuh — closest-hit / any-hit BVH traversal and the two shape tests, one thread per ray.
//
// Behavioural spec (what must match the reference bit for bit, SURVEY.md §10):
//   ray preparation  src/ray.jl:25-29, src/accel/bvh.jl:217-219, src/bounds.jl:169-175
//   slab test        src/bounds.jl:180-200   (SLAB = 0 literal, incl. the loose y far bound; SLAB = 1 standard)
//   traversal order  src/accel/bvh.jl:221-257 / 266-298  (near child by sign of d[split_axis], far child pushed)
//   triangle         src/shapes/triangle_mesh.jl:187-218, 245-273 (watertight shear test, FP64 only if ALL edges are 0)
//   sphere           src/shapes/sphere.jl:39-75, 125-191
// Layout: 32-byte nodes fetched as two 128-bit loads, 48-byte primitive records as three; a 64-entry per-thread stack
// (the reference's `zeros(Int32, 64)`), which the compiler keeps in local memory (L1-resident near its top).
#pragma once
#include "device_common.cuh"

struct RayPrep {            // quantities that depend on the ray only
    float3 o, d, inv;
    bool nx, ny, nz;
    int kz;                 // permutation of the triangle test
    float Sx, Sy, Sz;       // shear
    float mx, my, mz;       // SLAB 2: per-axis slack of the conservative interval, in units of t
    float mmax;             // max(mx, my, mz)
    bool any_zero;          // a direction component is 0: 1/d is Inf, slab products may be NaN - no shortcuts for this ray
    // thresholds of slab_child_fast; +Inf for an any_zero ray, which makes both of its verdicts false (-> full test)
    float fast_reject;      // 2 * mmax
    float fast_behind;      // mmax
    float fast_accept;      // 0
};

// Spatial slack of the conservative box test (SLAB 2), relative to the largest coordinate in play: 2^-17 ~ 7.6e-6,
// i.e. ~64 float ULPs - far above the rounding of the slab products and of the watertight triangle test, far below
// any triangle size.
#define TR_GUARD_REL 7.62939453125e-6f
#define TR_NODE_SPHERE_BELOW 0x20000000u   // device-side node meta bit 29, set at upload
#define TR_NODE_COUNT_MASK 0x1FFFFFFFu

__device__ __forceinline__ RayPrep prepare_ray(float3 o, float3 d, float scene_scale = 0.0f) {
    RayPrep r;
    // check_direction!: -0.0 -> +0.0 (x ≈ 0f0 is x == 0)
    if (d.x == 0.0f) d.x = 0.0f;
    if (d.y == 0.0f) d.y = 0.0f;
    if (d.z == 0.0f) d.z = 0.0f;
    r.o = o; r.d = d;
    r.inv = f3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
    r.nx = d.x < 0.0f; r.ny = d.y < 0.0f; r.nz = d.z < 0.0f;
    // _to_ray_coordinate_space: kz = first argmax |d|
    float ax = fabsf(d.x), ay = fabsf(d.y), az = fabsf(d.z);
    int kz = 0; float am = ax;
    if (ay > am) { kz = 1; am = ay; }
    if (az > am) { kz = 2; }
    r.kz = kz;
    float dx, dy, dz;
    if (kz == 0)      { dx = d.y; dy = d.z; dz = d.x; }
    else if (kz == 1) { dx = d.z; dy = d.x; dz = d.y; }
    else              { dx = d.x; dy = d.y; dz = d.z; }
    float denom = 1.0f / dz;
    r.Sx = -dx * denom; r.Sy = -dy * denom; r.Sz = denom;
    const float slack = TR_GUARD_REL * fmaxf(scene_scale, fmaxf(fabsf(o.x), fmaxf(fabsf(o.y), fabsf(o.z))));
    r.mx = slack * fabsf(r.inv.x); r.my = slack * fabsf(r.inv.y); r.mz = slack * fabsf(r.inv.z);
    r.mmax = fmaxf(r.mx, fmaxf(r.my, r.mz));
    r.any_zero = (d.x == 0.0f) | (d.y == 0.0f) | (d.z == 0.0f);
    r.fast_reject = r.any_zero ? TR_INF : 2.0f * r.mmax;
    r.fast_behind = r.any_zero ? TR_INF : r.mmax;
    r.fast_accept = r.any_zero ? TR_INF : 0.0f;
    return r;
}

// SLAB 0: the reference's test, literally (bounds.jl:180-200; line 191 keeps the LARGER y far bound, Q26).
// SLAB 1: the textbook test. NOT hit-equivalent to the reference (it drops rays grazing zero-thickness boxes): kept
//         only as a measured comparison, never a default.
// SLAB 2: "guarded": a node is entered iff the reference's test accepts it AND a conservative interval test (every
//         slab interval widened by the slack r.m*, NaN-transparent) cannot prove that the ray segment (0, t_max] misses
//         the box.  The visited set is a subset of the reference's, in the same order; a node is skipped only when
//         the ray provably stays clear of everything inside it, so hits, ties and t are the reference's.
// The guard is switched off (literal test only) for nodes whose subtree holds an analytic sphere
// (TR_NODE_SPHERE_BELOW): the reference's float32 quadratic (sphere.jl:39-54) is ill-conditioned for a small sphere
// seen from far away - b*b - 4ac cancels catastrophically and rays passing up to ~|o|^2 eps / 2r OUTSIDE the sphere
// still "hit" it at t ~ -b/2a.  The reference reports those hits (its loose box test lets the ray into the node), so
// the guarded variant must too; no fixed slack bounds that error.  Triangles have no such problem: the watertight
// test's error is a few ULPs of the coordinates.
template <int SLAB>
__device__ __forceinline__ bool slab_test(const float4 n0, const float4 n1, const RayPrep& r, float tmax) {
    // bmin = (n0.x, n0.y, n0.z), bmax = (n0.w, n1.x, n1.y)
    const float ax0 = ((r.nx ? n0.w : n0.x) - r.o.x) * r.inv.x;
    const float ax1 = ((r.nx ? n0.x : n0.w) - r.o.x) * r.inv.x;
    const float ay0 = ((r.ny ? n1.x : n0.y) - r.o.y) * r.inv.y;
    const float ay1 = ((r.ny ? n0.y : n1.x) - r.o.y) * r.inv.y;
    const float az0 = ((r.nz ? n1.y : n0.z) - r.o.z) * r.inv.z;
    const float az1 = ((r.nz ? n0.z : n1.y) - r.o.z) * r.inv.z;
    if (SLAB == 2 && !(__float_as_uint(n1.w) & TR_NODE_SPHERE_BELOW)) {
        // fmaxf / fminf drop NaNs (0 * Inf on an axis the ray is parallel to), so such an axis never rejects
        const float t_enter = fmaxf(fmaxf(ax0 - r.mx, ay0 - r.my), az0 - r.mz);
        const float t_exit = fminf(fminf(ax1 + r.mx, ay1 + r.my), az1 + r.mz);
        if (t_enter > t_exit || t_exit < 0.0f || t_enter > tmax + fabsf(tmax) * TR_GUARD_REL) return false;
    }
    float tx_min = ax0, tx_max = ax1;
    if (tx_min > ay1 || ay0 > tx_max) return false;
    if (ay0 > tx_min) tx_min = ay0;
    if (SLAB == 1) { if (ay1 < tx_max) tx_max = ay1; }
    else           { if (ay1 > tx_max) tx_max = ay1; }
    if (tx_min > az1 || az0 > tx_max) return false;
    if (az0 > tx_min) tx_min = az0;
    if (az1 < tx_max) tx_max = az1;
    return tx_min < tmax && tx_max > 0.0f;
}

// Watertight triangle test. a, b, c are the primitive record's float4s (xyz = vertices).
__device__ __forceinline__ bool triangle_test(const float4 a, const float4 b, const float4 c, const RayPrep& r, float tmax,
                                              float& t_hit, float& b0, float& b1, float& b2) {
    float X0, Y0, Z0, X1, Y1, Z1, X2, Y2, Z2;
    {
        float qx = a.x - r.o.x, qy = a.y - r.o.y, qz = a.z - r.o.z;     // (v - o), then permuted
        float px, py, pz;
        if (r.kz == 0) { px = qy; py = qz; pz = qx; } else if (r.kz == 1) { px = qz; py = qx; pz = qy; } else { px = qx; py = qy; pz = qz; }
        X0 = px + r.Sx * pz; Y0 = py + r.Sy * pz; Z0 = pz + 0.0f;
    }
    {
        float qx = b.x - r.o.x, qy = b.y - r.o.y, qz = b.z - r.o.z;
        float px, py, pz;
        if (r.kz == 0) { px = qy; py = qz; pz = qx; } else if (r.kz == 1) { px = qz; py = qx; pz = qy; } else { px = qx; py = qy; pz = qz; }
        X1 = px + r.Sx * pz; Y1 = py + r.Sy * pz; Z1 = pz + 0.0f;
    }
    {
        float qx = c.x - r.o.x, qy = c.y - r.o.y, qz = c.z - r.o.z;
        float px, py, pz;
        if (r.kz == 0) { px = qy; py = qz; pz = qx; } else if (r.kz == 1) { px = qz; py = qx; pz = qy; } else { px = qx; py = qy; pz = qz; }
        X2 = px + r.Sx * pz; Y2 = py + r.Sy * pz; Z2 = pz + 0.0f;
    }
    float e0 = X1 * Y2 - Y1 * X2;
    float e1 = X2 * Y0 - Y2 * X0;
    float e2 = X0 * Y1 - Y0 * X1;
    if (e0 == 0.0f && e1 == 0.0f && e2 == 0.0f) {
        e0 = (float)((double)X1 * (double)Y2 - (double)Y1 * (double)X2);
        e1 = (float)((double)X2 * (double)Y0 - (double)Y2 * (double)X0);
        e2 = (float)((double)X0 * (double)Y1 - (double)Y0 * (double)X1);
    }
    if ((e0 < 0.0f || e1 < 0.0f || e2 < 0.0f) && (e0 > 0.0f || e1 > 0.0f || e2 > 0.0f)) return false;
    float det = (e0 + e1) + e2;
    if (det == 0.0f) return false;
    float ts = ((e0 * Z0) * r.Sz + (e1 * Z1) * r.Sz) + (e2 * Z2) * r.Sz;
    if (det < 0.0f && (ts >= 0.0f || ts < tmax * det)) return false;
    if (det > 0.0f && (ts <= 0.0f || ts > tmax * det)) return false;
    float inv_det = 1.0f / det;
    b0 = e0 * inv_det; b1 = e1 * inv_det; b2 = e2 * inv_det;
    t_hit = ts * inv_det;
    return true;
}

struct SphereHitInfo { float t; float3 p; float phi; };

__device__ __forceinline__ float3 sphere_refine(float3 p, float radius) {
    float f = radius / length3(f3s(0.0f) - p);
    p = p * f;
    if (p.x == 0.0f && p.y == 0.0f) p = f3(1e-6f * radius, p.y, p.z);
    return p;
}
__device__ __forceinline__ float sphere_phi(float3 p) {
    float phi = atan2f(p.y, p.x);
    if (phi < 0.0f) phi += 2.0f * TR_PI;
    return phi;
}
__device__ __forceinline__ bool sphere_clipped(const DeviceSphere& s, float3 p, float phi) {
    return (s.z_min > -s.radius && p.z < s.z_min) || (s.z_max < s.radius && p.z > s.z_max) || phi > s.phi_max;
}
static __device__ __noinline__ bool sphere_test(const DeviceSphere& s, float3 ro, float3 rd, float tmax, SphereHitInfo& h) {
    float3 o = xform_point(s.inv_m, ro);
    float3 d = xform_vector(s.inv_m, rd);
    float nd = length3(d), no = length3(o);
    float a = nd * nd;
    float b = dot3(2.0f * o, d);
    float c = no * no - s.radius * s.radius;
    float disc = b * b - (4.0f * a) * c;
    if (disc < 0.0f) return false;
    float rdisc = sqrtf(disc);
    float q = -0.5f * (b + (b < 0.0f ? -rdisc : rdisc));
    float t0 = q / a, t1 = c / q;
    if (t0 > t1) { float tmp = t0; t0 = t1; t1 = tmp; }
    if (t0 > tmax || t1 < 0.0f) return false;
    if (t0 < 0.0f) t0 = t1;                                   // no t_max re-check (Q12)
    h.t = t0;
    h.p = sphere_refine(o + d * t0, s.radius);
    h.phi = sphere_phi(h.p);
    if (sphere_clipped(s, h.p, h.phi)) {
        h.t = t1;
        h.p = sphere_refine(o + d * t1, s.radius);
        h.phi = sphere_phi(h.p);
        if (sphere_clipped(s, h.p, h.phi)) return false;
    }
    return true;
}

#define TR_PRIM_SPHERE_BIT 0x80000000u
#define TR_PRIM_DEGENERATE_BIT 0x40000000u
#define TR_PRIM_LAST_BIT 0x20000000u        // last primitive of its BVH leaf (set at upload; used by the pair-node walk)
#define TR_PRIM_INDEX_MASK 0x1FFFFFFFu
#define TR_STACK_SIZE 64
#define TR_WALK_PAIR (-1)     // "walk" selector of the kernels: 0 reference loop, -1 pair nodes, 4..32 batched leaves
#ifndef TR_PARK_MAX
#define TR_PARK_MAX 12      // a leaf slot opens as soon as this many lanes of the warp are parked on a leaf
#endif

struct HitRecord {
    uint32_t prim;      // BVH-ordered primitive index + 1, 0 = miss
    float t, b0, b1;
};

// Returns true when something was hit. ANY: stops at the first accepted primitive (intersect_p).
// The loop is the reference's (bvh.jl:221-257): box-test the current node; leaf -> test its primitives in order, each
// accepted closest hit shrinks t_max; interior -> near child next (sign of d[split_axis]), far child pushed untested.
// Measured and rejected on B200 (profiles/r1_experiments.md): box-testing both children at their parent (0.7x), a
// min/max reformulation of the slab test with fewer instructions (0.75-0.98x), persistent warps with dynamic ray
// fetch (0.85x, kept below as option "persist"), a "while-while" loop whose lanes meet before testing primitives (0.32x:
// lanes standing on a leaf wait for the longest box-test walk of the warp), prefetching the pushed far child (0.98x),
// keeping the first 12 / 16 / 24 stack entries in shared memory (0.86-0.90x).
template <int SLAB, bool ANY, bool COUNT>
__device__ __forceinline__ bool traverse(const DeviceScene& sc, float3 o, float3 d, float tmax, HitRecord& out,
                                         unsigned long long* counters, int* error_flag) {
    out.prim = 0; out.t = tmax; out.b0 = 0.0f; out.b1 = 0.0f;
    if (sc.n_nodes == 0) return false;
    const RayPrep r = prepare_ray(o, d, sc.scene_scale);
    uint32_t stack[TR_STACK_SIZE];
    int sp = 0;
    uint32_t cur = 0;
    unsigned n_nodes = 0, n_prims = 0;
    bool found = false;
    for (;;) {
        const float4 n0 = __ldg(&sc.nodes[2 * cur]);
        const float4 n1 = __ldg(&sc.nodes[2 * cur + 1]);
        if (COUNT) n_nodes++;
        bool descend = false;
        if (slab_test<SLAB>(n0, n1, r, tmax)) {
            const uint32_t offset = __float_as_uint(n1.z), meta = __float_as_uint(n1.w);
            const uint32_t count = meta & TR_NODE_COUNT_MASK;
            if ((meta >> 30) == 3u) {     // leaf (a zero-primitive leaf has invalid bounds and never gets here, Q16/Q17)
                for (uint32_t i = 0; i < count; ++i) {
                    const uint32_t pi = offset + i;
                    const float4 a = __ldg(&sc.prims[3 * pi]);
                    const uint32_t tag = __float_as_uint(a.w);
                    if (COUNT) n_prims++;
                    if ((tag & ~TR_PRIM_LAST_BIT) == 0u) {
                        const float4 b = __ldg(&sc.prims[3 * pi + 1]);
                        const float4 c = __ldg(&sc.prims[3 * pi + 2]);
                        float t, b0, b1, b2;
                        if (triangle_test(a, b, c, r, tmax, t, b0, b1, b2)) {
                            if (ANY) { found = true; goto done; }
                            tmax = t; found = true;
                            out.prim = pi + 1; out.t = t; out.b0 = b0; out.b1 = b1;
                        }
                    } else if (tag & TR_PRIM_SPHERE_BIT) {
                        SphereHitInfo sh;
                        if (sphere_test(sc.spheres[tag & TR_PRIM_INDEX_MASK], r.o, r.d, tmax, sh)) {
                            if (ANY) { found = true; goto done; }
                            tmax = sh.t; found = true;
                            out.prim = pi + 1; out.t = sh.t; out.b0 = 0.0f; out.b1 = 0.0f;
                        }
                    }   // degenerate triangles (is_degenerate, triangle_mesh.jl:65-68) never hit
                }
            } else {
                const uint32_t axis = meta >> 30;
                const bool neg = axis == 0 ? r.nx : (axis == 1 ? r.ny : r.nz);
                if (sp >= TR_STACK_SIZE) { if (error_flag) *error_flag = 1; goto done; }
                if (neg) { stack[sp++] = cur + 1; cur = offset; }
                else     { stack[sp++] = offset; cur = cur + 1; }
                descend = true;
            }
        }
        if (!descend) {
            if (sp == 0) break;
            cur = stack[--sp];
        }
    }
done:
#ifdef TR_DEBUG_MAXNODES      // debugging aid: prims_tested becomes the LARGEST node count of any ray
    if (COUNT && counters) { atomicAdd(&counters[0], (unsigned long long)n_nodes); atomicMax(&counters[1], (unsigned long long)n_nodes); }
#else
    if (COUNT && counters) { atomicAdd(&counters[0], (unsigned long long)n_nodes); atomicAdd(&counters[1], (unsigned long long)n_prims); }
#endif
    return found;
}

// ------------------------------------------------------------------ pair-node traversal
// The reference walk (traverse<>() above) fetches and box-tests ONE node per iteration; every far child is pushed
// untested and most of them fail their test when popped.  ncu (profiles/r2_extend_source_base.txt): per iteration ~98
// instructions, 23-27 % of them stack push / pop bookkeeping at 13-19 of 32 lanes, and a dependent 32-byte fetch for every
// tested node.  The pair layout stores, in every interior node, the boxes of its TWO children (64 bytes, 4 x 128-bit
// loads issued together), so one fetch serves both box tests, which are independent and overlap in the pipeline:
//   * the near child (sign of d[split_axis], as the reference) is entered right away when its test passes;
//   * the far child's test is split: every condition of the reference's test but one is independent of t_max and is
//     evaluated NOW - a far child failing those is never pushed, it would fail when popped as well; one passing them
//     is pushed together with its entry distance tx_min, and the t_max-dependent condition (tx_min < t_max,
//     bounds.jl:199) is evaluated with the t_max of the moment it is popped, which is when the reference tests it -
//     a register compare, no fetch.
// The set of nodes whose primitives are tested, their order, and every t_max update are exactly those of the
// reference walk, so hits, tie-breaks and t are bit-identical (tests/test_gpu_parity.py runs both walks against the
// oracle).  Leaves need no node of their own: a child reference is either a pair index or the offset of the leaf's first
// primitive, and the primitive records carry a "last of its leaf" bit.  Stack: entries {ref, tx_min}, top of stack in
// registers so a pop never waits for local memory; it holds only box-hit nodes, so it is never deeper than the
// reference's (which overflows - BoundsError - beyond 64 pending nodes, bvh.jl:222; here that is reported as an error
// only if 64 box-HIT nodes are pending).
#define TR_REF_LEAF 0x80000000u
#define TR_REF_SPHERE_BELOW 0x40000000u
#define TR_REF_INDEX_MASK 0x3FFFFFFFu

// One child's box test WITHOUT its t_max condition: the reference's verdict (SLAB 0) or reference AND conservative
// guard (SLAB 2) for the ray (0, inf); tx_min_out is the reference's entry distance - the node is entered iff this
// returns true and tx_min_out < t_max (bounds.jl:199) with the t_max of the moment the reference would test it.
// Branch-free on purpose: the two children of a pair are tested back to back and their instruction streams interleave.
template <int SLAB>
__device__ __forceinline__ bool slab_child(const float4 n0, const float4 n1, const RayPrep& r, float& tx_min_out) {
    const float ax0 = ((r.nx ? n0.w : n0.x) - r.o.x) * r.inv.x;
    const float ax1 = ((r.nx ? n0.x : n0.w) - r.o.x) * r.inv.x;
    const float ay0 = ((r.ny ? n1.x : n0.y) - r.o.y) * r.inv.y;
    const float ay1 = ((r.ny ? n0.y : n1.x) - r.o.y) * r.inv.y;
    const float az0 = ((r.nz ? n1.y : n0.z) - r.o.z) * r.inv.z;
    const float az1 = ((r.nz ? n0.z : n1.y) - r.o.z) * r.inv.z;
    bool ok = true;
    if (SLAB == 2) {
        // conservative interval test (NaN-transparent); its t_max part is implied by the reference's tx_min < t_max
        const float t_enter = fmaxf(fmaxf(ax0 - r.mx, ay0 - r.my), az0 - r.mz);
        const float t_exit = fminf(fminf(ax1 + r.mx, ay1 + r.my), az1 + r.mz);
        const bool guard_miss = (t_enter > t_exit) | (t_exit < 0.0f);
        ok = !guard_miss | ((__float_as_uint(n1.z) & TR_REF_SPHERE_BELOW) != 0u);
    }
    // bounds.jl:180-200, literally (Q26: the y far bound keeps the LARGER value), all compares false on NaN
    ok &= !((ax0 > ay1) | (ay0 > ax1));
    float tx_min = ay0 > ax0 ? ay0 : ax0;
    float tx_max = ay1 > ax1 ? ay1 : ax1;
    ok &= !((tx_min > az1) | (az0 > tx_max));
    tx_min = az0 > tx_min ? az0 : tx_min;
    tx_max = az1 < tx_max ? az1 : tx_max;
    ok &= tx_max > 0.0f;
    tx_min_out = tx_min;
    return ok;               // the caller adds the one t_max-dependent condition: tx_min < t_max
}

// Fast three-way classification of one child's box test (SLAB 2 only).  With a0 = entry and a1 = exit distances of the
// three slabs (the same six products the reference forms), t_enter = max a0 and t_exit = min a1 (no NaN in play):
//   * ACCEPT when t_enter <= t_exit and t_exit > 0 - the textbook test on the reference's own numbers.  Every rejecting
//     comparison of the reference's test (bounds.jl:186-199, incl. the loose y far bound) implies t_enter > t_exit or
//     t_exit <= 0, so the reference accepts too, with tx_min == t_enter; the guard's interval is this one widened, so it
//     accepts as well.  Hence exactly what slab_child<2> returns.
//   * REJECT when the interval is empty by more than twice the largest slack, or ends before -slack: then the guard's
//     widened interval is empty / behind the origin as well, and slab_child<2> returns false (not used below analytic
//     spheres, where the guard is off).
//   * otherwise UNDECIDED (grazing within the slack band, NaN boxes): the caller evaluates slab_child<2> in full.
// About 26 instructions per child instead of 44; the undecided band is a few rays in a million box tests.
// The kernels are bound by the ALU pipe (ncu: 68 % against 22 % on the FMA pipe), so this form avoids what it can there:
// no selects by the direction's sign (1/d < 0 swaps the two products of an axis, so entry = min, exit = max of the pair -
// the same six numbers, hence the same t_enter bits), and the any_zero exclusion is folded into per-ray thresholds
// instead of being re-derived from the direction every iteration (predicates do not survive the loop).
__device__ __forceinline__ void slab_child_fast(const float4 n0, const float4 n1, const RayPrep& r, float& t_enter_out, bool& accept, bool& reject) {
    const float x0 = (n0.x - r.o.x) * r.inv.x, x1 = (n0.w - r.o.x) * r.inv.x;
    const float y0 = (n0.y - r.o.y) * r.inv.y, y1 = (n1.x - r.o.y) * r.inv.y;
    const float z0 = (n0.z - r.o.z) * r.inv.z, z1 = (n1.y - r.o.z) * r.inv.z;
    const float t_enter = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fminf(z0, z1));
    const float t_exit = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fmaxf(z0, z1));
    accept = (t_enter <= t_exit) & (t_exit > r.fast_accept);
    reject = (((t_enter - t_exit) > r.fast_reject) | (t_exit < -r.fast_behind)) & ((__float_as_uint(n1.z) & TR_REF_SPHERE_BELOW) == 0u);
    t_enter_out = t_enter;
}

// both children of a pair: static verdicts s0, s1 and entry distances t0, t1 (see slab_child)
template <int SLAB>
__device__ __forceinline__ void slab_children(const float4 q0, const float4 q1, const float4 q2, const float4 q3, const RayPrep& r,
                                              bool& s0, bool& s1, float& t0, float& t1) {
    if (SLAB == 2) {
        bool a0, r0, a1, r1;
        slab_child_fast(q0, q1, r, t0, a0, r0);
        slab_child_fast(q2, q3, r, t1, a1, r1);
        if ((a0 | r0) & (a1 | r1)) { s0 = a0; s1 = a1; return; }
    }
    s0 = slab_child<SLAB>(q0, q1, r, t0);
    s1 = slab_child<SLAB>(q2, q3, r, t1);
}

template <int SLAB, bool ANY, bool COUNT>
__device__ __forceinline__ bool traverse_pair(const DeviceScene& sc, float3 o, float3 d, float tmax, HitRecord& out,
                                              unsigned long long* counters, int* error_flag) {
    out.prim = 0; out.t = tmax; out.b0 = 0.0f; out.b1 = 0.0f;
    if (sc.n_nodes == 0) return false;
    const RayPrep r = prepare_ray(o, d, sc.scene_scale);
    unsigned n_nodes = 1, n_prims = 0;
    bool found = false;
    uint32_t item;
    {   // the root's own box (bvh.jl:224): the one node that is not somebody's child
        const float4 n0 = __ldg(&sc.nodes[0]), n1 = __ldg(&sc.nodes[1]);
        if (!slab_test<SLAB>(n0, n1, r, tmax)) { item = 0; goto done; }
        item = sc.root_ref;
    }
    {
    uint2 stack[TR_STACK_SIZE];
    uint2 tos = make_uint2(0u, 0u);
    int sp = 0;
    unsigned signs = (r.nx ? 1u : 0u) | (r.ny ? 2u : 0u) | (r.nz ? 4u : 0u);
    asm volatile("" : "+r"(signs));       // keep it in a register: ptxas otherwise re-derives it from d every iteration (7 ALU instructions)
    const bool cull_far = sc.n_spheres == 0;
    for (;;) {
        if (item & TR_REF_LEAF) {
            uint32_t pi = item & TR_REF_INDEX_MASK;
            for (;; ++pi) {
                const float4 a = __ldg(&sc.prims[3 * pi]);
                const uint32_t tag = __float_as_uint(a.w);
                if (COUNT) n_prims++;
                if ((tag & ~TR_PRIM_LAST_BIT) == 0u) {
                    const float4 b = __ldg(&sc.prims[3 * pi + 1]);
                    const float4 c = __ldg(&sc.prims[3 * pi + 2]);
                    float t, b0, b1, b2;
                    if (triangle_test(a, b, c, r, tmax, t, b0, b1, b2)) {
                        found = true;
                        if (ANY) goto done;
                        tmax = t;
                        out.prim = pi + 1; out.t = t; out.b0 = b0; out.b1 = b1;
                    }
                } else if (tag & TR_PRIM_SPHERE_BIT) {
                    SphereHitInfo sh;
                    if (sphere_test(sc.spheres[tag & TR_PRIM_INDEX_MASK], r.o, r.d, tmax, sh)) {
                        found = true;
                        if (ANY) goto done;
                        tmax = sh.t;
                        out.prim = pi + 1; out.t = sh.t; out.b0 = 0.0f; out.b1 = 0.0f;
                    }
                }
                if (tag & TR_PRIM_LAST_BIT) break;
            }
        } else {
            const float4* np = sc.pairs + 4u * (item & TR_REF_INDEX_MASK);
            const float4 q0 = __ldg(np), q1 = __ldg(np + 1), q2 = __ldg(np + 2), q3 = __ldg(np + 3);
            if (COUNT) n_nodes += 2;
            float t0, t1;
            bool s0, s1;
            slab_children<SLAB>(q0, q1, q2, q3, r, s0, s1, t0, t1);
            const bool neg = (signs & __float_as_uint(q1.w)) != 0u;      // near child = second child iff d[axis] < 0 (q1.w = 1 << axis)
            const uint32_t ref0 = __float_as_uint(q1.z), ref1 = __float_as_uint(q3.z);
            const float near_t = neg ? t1 : t0, far_t = neg ? t0 : t1;
            const bool near_hit = (neg ? s1 : s0) & (near_t < tmax);               // tested now, as the reference does
            const bool far_static = neg ? s0 : s1;                                // tested when popped: t_max may differ
            const uint32_t near_ref = neg ? ref1 : ref0, far_ref = neg ? ref0 : ref1;
            if (near_hit) {
                item = near_ref;
                // Early cull of the far child: a triangle hit never raises t_max by more than rounding (t = ts / det
                // with ts <= t_max * det: 3 roundings), so a far child beyond t_max (1 + 1e-3) can never pass when
                // popped.  An analytic sphere CAN raise t_max (Q12: from inside, the far root is reported without
                // re-checking t_max, sphere.jl:137-149), so scenes with spheres keep every statically hit far child.
                if (far_static & (cull_far ? !(far_t > tmax + fabsf(tmax) * 1e-3f) : true)) {
                    if (sp >= TR_STACK_SIZE) { if (error_flag) *error_flag = 1; goto done; }
                    stack[sp++] = tos;
                    tos = make_uint2(far_ref, __float_as_uint(far_t));
                }
                continue;
            }
            const bool far_hit = far_static & (far_t < tmax);
            if (far_hit) { item = far_ref; continue; }
        }
        // pop the next pending node that the (shrunken) t_max still lets in
        for (;;) {
            if (sp == 0) goto done;
            item = tos.x;
            const float t_in = __uint_as_float(tos.y);
            tos = stack[--sp];
            if (t_in < tmax) break;
        }
    }
    }
done:
    if (COUNT && counters) { atomicAdd(&counters[0], (unsigned long long)n_nodes); atomicAdd(&counters[1], (unsigned long long)n_prims); }
    return found;
}

// ------------------------------------------------------------------ any-hit walk on the shadow tree
// An any-hit query returns one bit and never changes t_max, so the reference's answer does not depend on the order in
// which its walk visits nodes: it is "some primitive passes triangle_test(r, t_max), and every reference-tree ancestor
// of that primitive passes the reference's box test".  traverse_shadow computes that bit on the shadow tree (an LBVH
// with one primitive per leaf, built at upload, DeviceScene::shadow_pairs), which costs about half the box tests of
// the reference tree, and ties every occluder it reports back to the reference tree with one exact check:
//   walk       every pair fetch tests both children with the guard of slab_child<2> (the interval widened by the slack
//              r.m*, with the t_max term of slab_test<2>); a child is entered iff that guard admits it.  t_max is fixed,
//              so every verdict is final when a child is pushed: the stack holds references only, nearer entry first.
//   candidate  a primitive whose triangle_test(r, t_max) passes (same RayPrep, same scene_scale as the reference walk);
//   check      the candidate triangle's own vertex box textbook-accepts: t_enter <= t_exit, t_exit > 0 and
//              t_enter < t_max, on the six products slab_child_fast forms.  Then the answer is "occluded".
//   end        no candidate: "not occluded"; only unconfirmed candidates: the reference walk (traverse_pair<2, true>)
//              answers, which is the answer without a shadow tree.
// Why this is the reference's bit:
//   * No false "not occluded".  The guarded reference walk already relies on the guard never rejecting a box that
//     contains the vertices of a triangle the ray passes (triangle_test) - the slack covers the rounding of the
//     watertight test; otherwise the guarded walk (the default) would differ from the literal one.  Shadow-tree boxes
//     are exact unions of their primitives' vertex boxes, so every reference candidate is admitted here all the way
//     down to its leaf and becomes a shadow-tree candidate.
//   * No false "occluded".  Every reference-tree ancestor box of a primitive contains the primitive's vertex box,
//     coordinate by coordinate (tests/test_shadow_tree_host.py checks it on the uploaded trees).  Subtracting o and
//     multiplying by inv are monotone under round-to-nearest, so on each axis the ancestor's two products bracket the
//     vertex box's: its textbook entry is <= the vertex box's entry and its exit is >= its exit.  A textbook ACCEPT
//     of the vertex box is therefore a textbook ACCEPT of every ancestor, the root included, with entry <= the vertex
//     box's entry < t_max.  By slab_child_fast's three-way argument that is the reference's literal and guarded
//     verdict with tx_min < t_max (so neither the far-child cull nor the pop test of traverse_pair drops it): the
//     reference walk reaches the candidate's leaf and tests the same triangle with the same t_max - "occluded".
//   * NaN never enters: the walk runs only for rays with a finite origin and a finite, non-zero 1/d on every axis
//     (the shadow tree's boxes hold no NaN: a NaN vertex means no shadow tree), so the min / max form of the six
//     products below is exactly the sign-selected form of slab_child<2>.  Other rays (a zero, tiny or non-finite
//     direction component: +Inf thresholds, never a fast accept) go to the reference walk directly.
// Deviation: the shadow tree is at most 64 levels deep (the upload refuses deeper ones), so this stack cannot
// overflow; a reference-tree overflow (64 box-hit pending far children) is reported only when the fallback runs.
#define TR_COUNTER_SHADOW_FALLBACKS 8      // offset of ST_SHADOW_FALLBACKS from `counters` (= stats + ST_NODES, context.hpp)

// the kernel instantiations that can walk the shadow tree: the guarded pair walk (the default), and the counting passes,
// which run the plain loop for closest hits but count the shadow walk the default path runs.  The launch picks them
// when the scene it passes has a shadow tree (shadow_launch_scene, context.hpp); every other launch runs a kernel
// without this walk, compiled exactly as before it existed
template <int SLAB, bool COUNT, int WAIT>
constexpr bool shadow_walk_capable = SLAB == 2 && (WAIT == TR_WALK_PAIR || COUNT);

// kept out of line: it runs for a few rays per thousand and would otherwise double the kernel's code
template <bool COUNT>
static __device__ __noinline__ bool shadow_fallback(const DeviceScene sc, float3 o, float3 d, float tmax,
                                                    unsigned long long* counters, int* error_flag) {
    if (counters) atomicAdd(&counters[TR_COUNTER_SHADOW_FALLBACKS], 1ull);
    HitRecord h;
    return traverse_pair<2, true, COUNT>(sc, o, d, tmax, h, counters, error_flag);
}

// textbook entry / exit of a box (lo.xyz, hi.xyz) for a ray with finite, non-zero inv (no NaN: min / max pick the
// same numbers as the sign-selected products)
__device__ __forceinline__ void slab_interval(float lx, float ly, float lz, float hx, float hy, float hz, const RayPrep& r,
                                              float slack_x, float slack_y, float slack_z, float& t_enter, float& t_exit) {
    const float x0 = (lx - r.o.x) * r.inv.x, x1 = (hx - r.o.x) * r.inv.x;
    const float y0 = (ly - r.o.y) * r.inv.y, y1 = (hy - r.o.y) * r.inv.y;
    const float z0 = (lz - r.o.z) * r.inv.z, z1 = (hz - r.o.z) * r.inv.z;
    t_enter = fmaxf(fmaxf(fminf(x0, x1) - slack_x, fminf(y0, y1) - slack_y), fminf(z0, z1) - slack_z);
    t_exit = fminf(fminf(fmaxf(x0, x1) + slack_x, fmaxf(y0, y1) + slack_y), fmaxf(z0, z1) + slack_z);
}

template <bool COUNT>
__device__ __forceinline__ bool traverse_shadow(const DeviceScene& sc, float3 o, float3 d, float tmax,
                                                unsigned long long* counters, int* error_flag) {
    const RayPrep r = prepare_ray(o, d, sc.scene_scale);
    const bool regular = isfinite(o.x) & isfinite(o.y) & isfinite(o.z) & isfinite(r.inv.x) & isfinite(r.inv.y) &
                         isfinite(r.inv.z) & (r.inv.x != 0.0f) & (r.inv.y != 0.0f) & (r.inv.z != 0.0f);
    if (!regular) return shadow_fallback<COUNT>(sc, o, d, tmax, counters, error_flag);
    const float tmax_guard = tmax + fabsf(tmax) * TR_GUARD_REL;        // slab_test<2>'s t_max term
    uint32_t stack[TR_STACK_SIZE];
    int sp = 0;
    uint32_t item = 0;                      // the root: pair 0
    unsigned n_nodes = 0, n_prims = 0;
    bool occluded = false, candidate = false;
    for (;;) {
        if (item & TR_REF_LEAF) {
            const uint32_t pi = item & TR_REF_INDEX_MASK;
            const float4 a = __ldg(&sc.prims[3 * pi]);
            if (COUNT) n_prims++;
            if ((__float_as_uint(a.w) & ~TR_PRIM_LAST_BIT) == 0u) {        // degenerate triangles never hit
                const float4 b = __ldg(&sc.prims[3 * pi + 1]), c = __ldg(&sc.prims[3 * pi + 2]);
                float t, b0, b1, b2;
                if (triangle_test(a, b, c, r, tmax, t, b0, b1, b2)) {
                    float t_enter, t_exit;
                    slab_interval(fminf(fminf(a.x, b.x), c.x), fminf(fminf(a.y, b.y), c.y), fminf(fminf(a.z, b.z), c.z),
                                  fmaxf(fmaxf(a.x, b.x), c.x), fmaxf(fmaxf(a.y, b.y), c.y), fmaxf(fmaxf(a.z, b.z), c.z), r,
                                  0.0f, 0.0f, 0.0f, t_enter, t_exit);
                    if ((t_enter <= t_exit) & (t_exit > 0.0f) & (t_enter < tmax)) { occluded = true; break; }
                    candidate = true;
                }
            }
        } else {
            const float4* np = sc.shadow_pairs + 4u * item;
            const float4 q0 = __ldg(np), q1 = __ldg(np + 1), q2 = __ldg(np + 2), q3 = __ldg(np + 3);
            if (COUNT) n_nodes += 2;
            float e0, x0, e1, x1;
            slab_interval(q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, r, r.mx, r.my, r.mz, e0, x0);
            slab_interval(q2.x, q2.y, q2.z, q2.w, q3.x, q3.y, r, r.mx, r.my, r.mz, e1, x1);
            const bool in0 = !((e0 > x0) | (x0 < 0.0f) | (e0 > tmax_guard));
            const bool in1 = !((e1 > x1) | (x1 < 0.0f) | (e1 > tmax_guard));
            const uint32_t ref0 = __float_as_uint(q1.z), ref1 = __float_as_uint(q3.z);
            if (in0 & in1) {
                const bool second_first = e1 < e0;
                stack[sp++] = second_first ? ref0 : ref1;
                item = second_first ? ref1 : ref0;
                continue;
            }
            if (in0 | in1) { item = in0 ? ref0 : ref1; continue; }
        }
        if (sp == 0) break;
        item = stack[--sp];
    }
    if (COUNT && counters) { atomicAdd(&counters[0], (unsigned long long)n_nodes); atomicAdd(&counters[1], (unsigned long long)n_prims); }
    if (occluded || !candidate) return occluded;
    return shadow_fallback<COUNT>(sc, o, d, tmax, counters, error_flag);
}

// ------------------------------------------------------------------ warp-synchronous traversal with batched leaves
// Same walk, same order, same tests as traverse<>() per ray - only WHEN a lane runs the primitive tests of a leaf changes.
// In the plain loop a warp executes the ~120-instruction triangle test whenever ANY of its lanes stands on a leaf;
// leaves are ~2 % of the node visits, so with 32 lanes about every second iteration pays for it with one or two lanes
// active (ncu round 1: 21 of 32 lanes on coherent primary rays, 12-15 on secondary rays).  Here the warp iterates in
// explicit lock step (one vote per iteration); a lane that reaches a leaf PARKS - it keeps the leaf pending and
// idles - until the warp opens a leaf slot: every WAIT-th iteration, or as soon as PARK_MAX lanes are parked, or when
// no lane is left traversing.  All parked lanes then run the primitive tests together.  A ray visits only ~1.6
// leaves, so parking adds a few idle iterations to a ~77-iteration walk, while the primitive tests run far less often
// and with many lanes.  Per-ray results are those of traverse<>(): node sequence, t_max updates and tie-breaks are
// unchanged (each lane still walks its own ray strictly in order).
// All 32 lanes of the warp must call this together; `valid == false` lanes only take part in the votes.
template <int SLAB, bool ANY, bool COUNT, int WAIT, int PARK_MAX>
__device__ __forceinline__ bool traverse_lb(const DeviceScene& sc, bool valid, float3 o, float3 d, float tmax, HitRecord& out,
                                            unsigned long long* counters, int* error_flag) {
    const unsigned full = 0xffffffffu;
    out.prim = 0; out.t = tmax; out.b0 = 0.0f; out.b1 = 0.0f;
    const RayPrep r = prepare_ray(o, d, sc.scene_scale);
    uint32_t stack[TR_STACK_SIZE];
    int sp = 0;
    uint32_t cur = 0;
    uint32_t leaf_off = 0, leaf_cnt = 0;          // pending leaf of this lane (leaf_cnt > 0: parked)
    unsigned n_nodes = 0, n_prims = 0;
    bool found = false;
    bool done = !valid || sc.n_nodes == 0;
    for (uint32_t it = 1;; ++it) {
        const unsigned m_trav = __ballot_sync(full, !done && leaf_cnt == 0u);
        const unsigned m_park = __ballot_sync(full, leaf_cnt != 0u);
        if ((m_trav | m_park) == 0u) break;
        const bool leaf_slot = m_trav == 0u || __popc(m_park) >= PARK_MAX || (it & (uint32_t)(WAIT - 1)) == 0u;
        if (leaf_cnt) {
            if (!leaf_slot) continue;                 // parked
            for (uint32_t i = 0; i < leaf_cnt; ++i) {
                const uint32_t pi = leaf_off + i;
                const float4 a = __ldg(&sc.prims[3 * pi]);
                const uint32_t tag = __float_as_uint(a.w);
                if (COUNT) n_prims++;
                if ((tag & ~TR_PRIM_LAST_BIT) == 0u) {
                    const float4 b = __ldg(&sc.prims[3 * pi + 1]);
                    const float4 c = __ldg(&sc.prims[3 * pi + 2]);
                    float t, b0, b1, b2;
                    if (triangle_test(a, b, c, r, tmax, t, b0, b1, b2)) {
                        found = true;
                        if (ANY) { done = true; break; }
                        tmax = t;
                        out.prim = pi + 1; out.t = t; out.b0 = b0; out.b1 = b1;
                    }
                } else if (tag & TR_PRIM_SPHERE_BIT) {
                    SphereHitInfo sh;
                    if (sphere_test(sc.spheres[tag & TR_PRIM_INDEX_MASK], r.o, r.d, tmax, sh)) {
                        found = true;
                        if (ANY) { done = true; break; }
                        tmax = sh.t;
                        out.prim = pi + 1; out.t = sh.t; out.b0 = 0.0f; out.b1 = 0.0f;
                    }
                }
            }
            leaf_cnt = 0;
            if (!done) { if (sp == 0) done = true; else cur = stack[--sp]; }
            continue;
        }
        if (done) continue;
        const float4 n0 = __ldg(&sc.nodes[2 * cur]);
        const float4 n1 = __ldg(&sc.nodes[2 * cur + 1]);
        if (COUNT) n_nodes++;
        if (slab_test<SLAB>(n0, n1, r, tmax)) {
            const uint32_t offset = __float_as_uint(n1.z), meta = __float_as_uint(n1.w);
            if ((meta >> 30) == 3u) {
                leaf_cnt = meta & TR_NODE_COUNT_MASK;
                leaf_off = offset;
                if (leaf_cnt) continue;
            } else {
                const uint32_t axis = meta >> 30;
                const bool neg = axis == 0 ? r.nx : (axis == 1 ? r.ny : r.nz);
                if (sp >= TR_STACK_SIZE) { if (error_flag) *error_flag = 1; done = true; continue; }
                if (neg) { stack[sp++] = cur + 1; cur = offset; }
                else     { stack[sp++] = offset; cur = cur + 1; }
                continue;
            }
        }
        if (sp == 0) done = true; else cur = stack[--sp];
    }
    if (COUNT && counters && valid) { atomicAdd(&counters[0], (unsigned long long)n_nodes); atomicAdd(&counters[1], (unsigned long long)n_prims); }
    return found;
}

// dispatch: WAIT == 0 is the plain per-thread loop.  All 32 lanes of a warp must call this together.
template <int SLAB, bool ANY, bool COUNT, int WAIT>
__device__ __forceinline__ bool traverse_any(const DeviceScene& sc, bool valid, float3 o, float3 d, float tmax, HitRecord& out,
                                             unsigned long long* counters, int* error_flag) {
    if (WAIT == 0 || WAIT == TR_WALK_PAIR) {
        if (!valid) { out.prim = 0; out.t = tmax; out.b0 = 0.0f; out.b1 = 0.0f; return false; }
        if (WAIT == TR_WALK_PAIR) return traverse_pair<SLAB == 1 ? 0 : SLAB, ANY, COUNT>(sc, o, d, tmax, out, counters, error_flag);
        return traverse<SLAB, ANY, COUNT>(sc, o, d, tmax, out, counters, error_flag);
    } else return traverse_lb<SLAB, ANY, COUNT, (WAIT > 0 ? WAIT : 1), TR_PARK_MAX>(sc, valid, o, d, tmax, out, counters, error_flag);
}

