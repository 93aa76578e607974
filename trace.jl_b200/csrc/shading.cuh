// shading.cuh — device-side hit-record construction, BSDF lobes, lights, sampling warps and the Halton sampler.
// Behavioural spec: SURVEY.md §10.4-10.5 (hit record) and §11 (lobes), i.e. the reference's
//   src/shapes/triangle_mesh.jl:125-185,220-242   src/shapes/sphere.jl:77-93,150-163   src/surface_interaction.jl:51-88,154-181
//   src/reflection/{bxdf,specular,lambertian,microfacet}.jl   src/materials/{bsdf,material}.jl
//   src/lights/{point,spot}.jl   src/Trace.jl:48-126   src/sampler/sampling.jl:43-76
// with its quirks (Q6 no eta^2 scaling, Q18, Q24 gating on the geometric normal, Q27 microfacet pdf).
#pragma once
#include "traverse.cuh"

enum : uint32_t { LB_REFLECTION = 1, LB_TRANSMISSION = 2, LB_DIFFUSE = 4, LB_GLOSSY = 8, LB_SPECULAR = 16, LB_ALL = 31 };
enum : int { LK_LAMBERT = 0, LK_SPEC_REFL = 1, LK_SPEC_TRANS = 2, LK_FRESNEL_SPEC = 3, LK_MICRO_REFL = 4, LK_MICRO_TRANS = 5,
             LK_OREN_NAYAR = 6 };

struct Interaction {
    float3 p, wo, ng, ns, dpdu;     // core.p, core.wo, core.n, shading.n, shading.∂p∂u
    uint32_t material;
};

struct Frame { float3 ss, ts, ns, ng; };   // BSDF frame, materials/bsdf.jl:37-50

struct Lobe {
    int kind;
    uint32_t type;
    float3 r, t;
    float eta_a, eta_b;
    int fresnel;            // 0 FresnelNoOp, 1 FresnelDielectric(fi, ft)
    float fi, ft;
    float ax, ay;           // Trowbridge-Reitz alphas; Oren-Nayar: A and B (microfacet.jl:12-18)
};
struct LobeSet { Lobe l[2]; int n; };

// ------------------------------------------------------------------ hit record
__device__ __forceinline__ void coordinate_system(float3 v1, float3& v2, float3& v3) {      // Trace.jl:139-146
    if (fabsf(v1.x) > fabsf(v1.y)) v2 = f3(-v1.z, 0.0f, v1.x) / sqrtf(v1.x * v1.x + v1.z * v1.z);
    else v2 = f3(0.0f, v1.z, -v1.y) / sqrtf(v1.y * v1.y + v1.z * v1.z);
    v3 = cross3(v1, v2);
}
__device__ __forceinline__ float3 face_forward(float3 n, float3 v) { return dot3(n, v) < 0.0f ? -n : n; }

// prim: 0-based BVH-ordered index of the winning primitive; (b0,b1,b2): its barycentrics (triangles);
// ray_d: the direction as intersect! leaves it (after check_direction!).
__device__ __forceinline__ Interaction build_interaction(const DeviceScene& sc, uint32_t prim, float3 ray_o, float3 ray_d,
                                                         float b0, float b1, float b2) {
    Interaction it;
    const float4 A = __ldg(&sc.prims[3 * prim]), B = __ldg(&sc.prims[3 * prim + 1]);
    const uint32_t tag = __float_as_uint(A.w);
    it.material = __float_as_uint(B.w);
    if (!(tag & TR_PRIM_SPHERE_BIT)) {
        const float4 C = __ldg(&sc.prims[3 * prim + 2]);
        const float3 p0 = xyz(A), p1 = xyz(B), p2 = xyz(C);
        const float3 dp13 = p0 - p2, dp23 = p1 - p2;
        // ∂p∂u for the default uv (0,0),(1,0),(1,1): δuv13 = (-1,-1), δuv23 = (0,-1), det = 1 (triangle_mesh.jl:125-141)
        const float3 dpdu = ((-1.0f) * dp13 - (-1.0f) * dp23) * 1.0f;
        it.p = (b0 * p0 + b1 * p1) + b2 * p2;
        it.wo = -ray_d;
        float3 ng = normalize3(cross3(dp13, dp23));
        float3 ns = ng;
        it.dpdu = dpdu;
        const float4 N0 = __ldg(&sc.tnorm[3 * prim]);
        const uint32_t flags = __float_as_uint(N0.w);
        if (flags & TRACE_TRI_HAS_NORMALS) {
            const float4 N1 = __ldg(&sc.tnorm[3 * prim + 1]), N2 = __ldg(&sc.tnorm[3 * prim + 2]);
            const float3 ns0 = normalize3((b0 * xyz(N0) + b1 * xyz(N1)) + b2 * xyz(N2));
            float3 ss = normalize3(dpdu);
            float3 ts = cross3(ns0, ss);
            if (dot3(ts, ts) > 0.0f) { ts = normalize3(ts); ss = cross3(ts, ns0); }
            else { coordinate_system(ns0, ss, ts); }
            ns = normalize3(cross3(ss, ts));
            if (flags & TRACE_TRI_FLIP) ns = ns * -1.0f;
            ng = face_forward(ng, ns);
            it.dpdu = ss;
        } else if (flags & TRACE_TRI_FLIP) {
            ng = -ng; ns = ng;
        }
        it.ng = ng; it.ns = ns;
    } else {
        const DeviceSphere& sp = sc.spheres[tag & TR_PRIM_INDEX_MASK];
        SphereHitInfo sh;
        sphere_test(sp, ray_o, ray_d, TR_INF, sh);          // same root as the accepted candidate (pure function of the ray)
        const float3 hp = sh.p;
        const float theta = acosf(clampf(hp.z / sp.radius, -1.0f, 1.0f));
        const float zr = sqrtf(hp.x * hp.x + hp.y * hp.y);
        const float inv_zr = 1.0f / zr;
        const float cos_phi = hp.x * inv_zr, sin_phi = hp.y * inv_zr;
        const float3 dpdu = f3(-sp.phi_max * hp.y, sp.phi_max * hp.x, 0.0f);
        const float3 dpdv = (sp.theta_max - sp.theta_min) * f3(hp.z * cos_phi, hp.z * sin_phi, -sp.radius * sinf(theta));
        float3 n = normalize3(cross3(dpdu, dpdv));
        if (sp.flip) n = n * -1.0f;
        it.p = xform_point(sp.m, hp);
        it.wo = normalize3(xform_vector(sp.m, -ray_d));
        it.ng = normalize3(xform_normal(sp.inv_m, n));
        it.ns = it.ng;
        it.dpdu = xform_vector(sp.m, dpdu);
    }
    return it;
}

__device__ __forceinline__ Frame make_frame(const Interaction& it) {
    Frame f;
    f.ng = it.ng; f.ns = it.ns;
    f.ss = normalize3(it.dpdu);
    f.ts = cross3(f.ns, f.ss);
    return f;
}
__device__ __forceinline__ float3 to_local(const Frame& f, float3 v) { return f3(dot3(v, f.ss), dot3(v, f.ts), dot3(v, f.ns)); }
__device__ __forceinline__ float3 to_world(const Frame& f, float3 v) {
    return f3((f.ss.x * v.x + f.ts.x * v.y) + f.ns.x * v.z, (f.ss.y * v.x + f.ts.y * v.y) + f.ns.y * v.z,
              (f.ss.z * v.x + f.ts.z * v.y) + f.ns.z * v.z);
}

// ------------------------------------------------------------------ lobes of a material (materials/material.jl)
__device__ __forceinline__ float3 clamp_spectrum(const float* c) {
    return f3(clampf(c[0], 0.0f, TR_INF), clampf(c[1], 0.0f, TR_INF), clampf(c[2], 0.0f, TR_INF));
}
__device__ __forceinline__ Lobe make_lobe(int kind, uint32_t type) {
    Lobe l;
    l.kind = kind; l.type = type; l.r = f3s(0.0f); l.t = f3s(0.0f); l.eta_a = 1.0f; l.eta_b = 1.0f;
    l.fresnel = 0; l.fi = 1.0f; l.ft = 1.0f; l.ax = 0.0f; l.ay = 0.0f;
    return l;
}
// multi = allow_multiple_lobes (false: Whitted, true: SPPM camera & photon passes)
__device__ __forceinline__ void material_lobes(const DeviceMaterial& m, bool multi, LobeSet& s) {
    s.n = 0;
    const float3 A = clamp_spectrum(m.a), B = clamp_spectrum(m.b);
    if (m.kind == TRACE_MAT_MATTE) {
        if (is_black3(A)) return;
        if (m.specular) {                // sigma == 0 -> Lambertian (material.jl:26-30)
            Lobe l = make_lobe(LK_LAMBERT, LB_DIFFUSE | LB_REFLECTION); l.r = A; s.l[s.n++] = l;
        } else {
            Lobe l = make_lobe(LK_OREN_NAYAR, LB_DIFFUSE | LB_REFLECTION); l.r = A; l.ax = m.alpha_u; l.ay = m.alpha_v; s.l[s.n++] = l;
        }
    } else if (m.kind == TRACE_MAT_MIRROR) {
        if (is_black3(A)) return;
        Lobe l = make_lobe(LK_SPEC_REFL, LB_SPECULAR | LB_REFLECTION); l.r = A; s.l[s.n++] = l;
    } else if (m.kind == TRACE_MAT_GLASS) {
        if (is_black3(A) && is_black3(B)) return;
        const bool spec = m.specular != 0u;
        if (spec && multi) {
            Lobe l = make_lobe(LK_FRESNEL_SPEC, LB_SPECULAR | LB_TRANSMISSION | LB_REFLECTION);
            l.r = A; l.t = B; l.eta_a = 1.0f; l.eta_b = m.eta; s.l[s.n++] = l;
            return;
        }
        if (!is_black3(A)) {
            Lobe l = spec ? make_lobe(LK_SPEC_REFL, LB_SPECULAR | LB_REFLECTION) : make_lobe(LK_MICRO_REFL, LB_REFLECTION | LB_GLOSSY);
            l.r = A; l.fresnel = 1; l.fi = 1.0f; l.ft = m.eta; l.ax = m.alpha_u; l.ay = m.alpha_v; s.l[s.n++] = l;
        }
        if (!is_black3(B)) {
            Lobe l = spec ? make_lobe(LK_SPEC_TRANS, LB_SPECULAR | LB_TRANSMISSION) : make_lobe(LK_MICRO_TRANS, LB_TRANSMISSION | LB_GLOSSY);
            l.t = B; l.eta_a = 1.0f; l.eta_b = m.eta; l.ax = m.alpha_u; l.ay = m.alpha_v; s.l[s.n++] = l;
        }
    } else {   // TRACE_MAT_PLASTIC
        if (!is_black3(A)) { Lobe l = make_lobe(LK_LAMBERT, LB_DIFFUSE | LB_REFLECTION); l.r = A; s.l[s.n++] = l; }
        if (is_black3(B)) return;
        Lobe l = make_lobe(LK_MICRO_REFL, LB_REFLECTION | LB_GLOSSY);
        l.r = B; l.fresnel = 1; l.fi = 1.5f; l.ft = 1.0f; l.ax = m.alpha_u; l.ay = m.alpha_u;
        s.l[s.n++] = l;
    }
}
__device__ __forceinline__ bool lobe_matches(const Lobe& l, uint32_t flags) { return (l.type & flags) == l.type; }
__device__ __forceinline__ int num_components(const LobeSet& s, uint32_t flags) {
    int n = 0;
    for (int i = 0; i < s.n; ++i) n += lobe_matches(s.l[i], flags) ? 1 : 0;
    return n;
}

// Julia's max(0f0, x) and min(x, 1f0): a NaN x stays NaN (fmaxf / fminf would return the other operand) and
// max(0f0, -0f0) is +0, as the reference computes them (the oracle's jl_max / jl_min)
__device__ __forceinline__ float jl_max0(float x) { return !(x <= 0.0f) ? x : 0.0f; }
__device__ __forceinline__ float jl_min1(float x) { return !(x >= 1.0f) ? x : 1.0f; }

// ------------------------------------------------------------------ local-frame helpers, Trace.jl:109-121
__device__ __forceinline__ float cos_th(float3 w) { return w.z; }
__device__ __forceinline__ float sin_th(float3 w) { return sqrtf(jl_max0(1.0f - w.z * w.z)); }
__device__ __forceinline__ float tan_th(float3 w) { return sin_th(w) / w.z; }
__device__ __forceinline__ float cos_ph(float3 w) { float s = sin_th(w); return s == 0.0f ? 1.0f : clampf(w.x / s, -1.0f, 1.0f); }
__device__ __forceinline__ float sin_ph(float3 w) { float s = sin_th(w); return s == 0.0f ? 1.0f : clampf(w.y / s, -1.0f, 1.0f); }
__device__ __forceinline__ bool same_hemi(float3 a, float3 b) { return a.z * b.z > 0.0f; }
__device__ __forceinline__ float sqr(float x) { return x * x; }
__device__ __forceinline__ float pow4f(float x) { double d = (double)x; d = d * d; return (float)(d * d); }

// ------------------------------------------------------------------ warps, Trace.jl:48-96
__device__ __forceinline__ float2 concentric_disk(float u0, float u1) {
    float x = 2.0f * u0 - 1.0f, y = 2.0f * u1 - 1.0f;
    if (x == 0.0f && y == 0.0f) return make_float2(0.0f, 0.0f);
    float r, th;
    if (fabsf(x) > fabsf(y)) { r = x; th = (y / x) * TR_PI / 4.0f; }
    else { r = y; th = TR_PI / 2.0f - (x / y) * TR_PI / 4.0f; }
    return make_float2(r * cosf(th), r * sinf(th));
}
__device__ __forceinline__ float3 cosine_hemisphere(float u0, float u1) {
    float2 d = concentric_disk(u0, u1);
    return f3(d.x, d.y, sqrtf(jl_max0(1.0f - d.x * d.x - d.y * d.y)));
}
__device__ __forceinline__ float3 uniform_sphere(float u0, float u1) {
    float z = 1.0f - 2.0f * u0;
    float r = sqrtf(jl_max0(1.0f - z * z));
    float phi = 2.0f * TR_PI * u1;
    return f3(r * cosf(phi), r * sinf(phi), z);
}
__device__ __forceinline__ float3 uniform_cone(float u0, float u1, float cmax) {
    float c = 1.0f - u0 + u0 * cmax;
    float s = sqrtf(1.0f - c * c);
    float phi = u1 * 2.0f * TR_PI;
    return f3(cosf(phi) * s, sinf(phi) * s, c);
}

// ------------------------------------------------------------------ Fresnel / refraction, reflection/bxdf.jl:52-95
__device__ __forceinline__ bool refract(float3 wi, float3 n, float eta, float3& wt) {
    float ci = dot3(n, wi);
    float s2i = jl_max0(1.0f - ci * ci);
    float s2t = (eta * eta) * s2i;
    if (s2t >= 1.0f) { wt = f3s(0.0f); return false; }
    float ct = sqrtf(1.0f - s2t);
    wt = (-eta) * wi + (eta * ci - ct) * n;
    return true;
}
__device__ __forceinline__ float fresnel_dielectric(float ci, float ei, float et) {
    ci = clampf(ci, -1.0f, 1.0f);
    if (ci <= 0.0f) { float t = ei; ei = et; et = t; ci = fabsf(ci); }
    float si = sqrtf(jl_max0(1.0f - ci * ci));
    float st = si * ei / et;
    if (st >= 1.0f) return 1.0f;
    float ct = sqrtf(jl_max0(1.0f - st * st));
    float rpar = (et * ci - ei * ct) / (et * ci + ei * ct);
    float rper = (ei * ci - et * ct) / (ei * ci + et * ct);
    return 0.5f * (rpar * rpar + rper * rper);
}
__device__ __forceinline__ float lobe_fresnel(const Lobe& l, float c) { return l.fresnel ? fresnel_dielectric(c, l.fi, l.ft) : 1.0f; }

// ------------------------------------------------------------------ Trowbridge-Reitz, reflection/microfacet.jl:53-201
__device__ __forceinline__ float tr_lambda(const Lobe& l, float3 w) {
    float th = fabsf(tan_th(w));
    if (isinf(th)) return 0.0f;
    float a = sqrtf(sqr(cos_ph(w)) * sqr(l.ax) + sqr(sin_ph(w)) * sqr(l.ay));
    return (-1.0f + sqrtf(1.0f + sqr(a * th))) / 2.0f;
}
__device__ __forceinline__ float tr_D(const Lobe& l, float3 w) {
    float t2 = sqr(tan_th(w));
    if (isinf(t2)) return 0.0f;
    float c4 = pow4f(w.z);
    float e = (sqr(cos_ph(w)) / sqr(l.ax) + sqr(sin_ph(w)) / sqr(l.ay)) * t2;
    return 1.0f / (TR_PI * l.ax * l.ay * c4 * sqr(1.0f + e));
}
__device__ __forceinline__ float tr_pdf(const Lobe& l, float3 wo, float3 wh) {
    return tr_D(l, wh) * (1.0f / (1.0f + tr_lambda(l, wo))) * fabsf(dot3(wo, wh)) / fabsf(wo.z);
}
__device__ __forceinline__ float2 tr_sample11(float cth, float u1, float u2) {
    if (cth > 0.9999f) {
        float r = sqrtf(u1 / (1.0f - u1));
        double phi = 6.28318530718 * (double)u2;
        return make_float2((float)((double)r * cos(phi)), (float)((double)r * sin(phi)));
    }
    float sth = sqrtf(jl_max0(1.0f - cth * cth));
    float tth = sth / cth;
    float a = 1.0f / tth;
    float g1 = 2.0f / (1.0f + sqrtf(1.0f + 1.0f / (a * a)));
    a = 2.0f * u1 / g1 - 1.0f;
    float tmp = 1.0f / (a * a - 1.0f);
    if (tmp > 1e10f) tmp = 1e10f;
    float b = tth, b2 = b * b;
    float d = sqrtf(jl_max0(b2 * (tmp * tmp) - (a * a - b2) * tmp));
    float x1 = b * tmp - d, x2 = b * tmp + d;
    float sx = (a < 0.0f || x2 > 1.0f / tth) ? x1 : x2;
    float s;
    if (u2 > 0.5f) { s = 1.0f; u2 = 2.0f * (u2 - 0.5f); } else { s = -1.0f; u2 = 2.0f * (0.5f - u2); }
    float z = (u2 * (u2 * (u2 * 0.27385f - 0.73369f) + 0.46341f)) / (u2 * (u2 * (u2 * 0.093073f + 0.309420f) - 1.0f) + 0.597999f);
    return make_float2(sx, s * z * sqrtf(1.0f + sx * sx));
}
__device__ __forceinline__ float3 tr_sample_wh(const Lobe& l, float3 wo, float u0, float u1) {
    bool flip = wo.z < 0.0f;
    float3 wi = flip ? -wo : wo;
    float3 ws = normalize3(f3(wi.x * l.ax, wi.y * l.ay, wi.z));
    float2 sl = tr_sample11(ws.z, u0, u1);
    float c = cos_ph(ws), s = sin_ph(ws);
    float tmp = c * sl.x - s * sl.y;
    sl.y = s * sl.x + c * sl.y;
    sl.x = tmp;
    sl.x *= l.ax; sl.y *= l.ay;
    float3 wh = normalize3(f3(-sl.x, -sl.y, 1.0f));
    return flip ? -wh : wh;
}

// ------------------------------------------------------------------ per-lobe f / pdf / sample_f (local frame)
__device__ __forceinline__ float3 lobe_f(const Lobe& l, float3 wo, float3 wi) {
    if (l.kind == LK_LAMBERT) return l.r * (1.0f / TR_PI);
    if (l.kind == LK_MICRO_REFL) {
        float co = fabsf(wo.z), ci = fabsf(wi.z);
        float3 wh = wi + wo;
        if (ci == 0.0f || co == 0.0f) return f3s(0.0f);
        if (is_black3(wh)) return f3s(0.0f);
        wh = normalize3(wh);
        float fr = lobe_fresnel(l, dot3(wi, face_forward(wh, f3(0.0f, 0.0f, 1.0f))));
        float G = 1.0f / (1.0f + tr_lambda(l, wo) + tr_lambda(l, wi));
        return l.r * tr_D(l, wh) * G * fr / (4.0f * ci * co);
    }
    if (l.kind == LK_MICRO_TRANS) {                    // microfacet.jl:280-305
        if (same_hemi(wo, wi)) return f3s(0.0f);
        const float co = wo.z, ci = wi.z;
        if (co == 0.0f || ci == 0.0f) return f3s(0.0f);
        const float eta = wo.z > 0.0f ? (l.eta_b / l.eta_a) : (l.eta_a / l.eta_b);
        float3 wh = normalize3(wo + wi * eta);
        if (wh.z < 0.0f) wh = -wh;
        const float d_o = dot3(wo, wh), d_i = dot3(wi, wh);
        if (d_o * d_i > 0.0f) return f3s(0.0f);
        const float fr = fresnel_dielectric(d_o, l.eta_a, l.eta_b);
        const float denom = d_o + eta * d_i;
        const float dd = tr_D(l, wh), dg = 1.0f / (1.0f + tr_lambda(l, wo) + tr_lambda(l, wi));
        const float v = fabsf(dd * dg * d_o * d_i * (eta * eta) * (1.0f * 1.0f) / (ci * co * (denom * denom)));   // factor = 1 (Q6)
        return ((f3s(1.0f) - f3s(fr)) * l.t) * v;
    }
    if (l.kind == LK_OREN_NAYAR) {                     // microfacet.jl:21-42
        const float si = sin_th(wi), so = sin_th(wo);
        float max_cos = 0.0f;
        if (si > 1e-4f && so > 1e-4f) max_cos = jl_max0(cos_ph(wi) * cos_ph(wo) + sin_ph(wi) * sin_ph(wo));
        float sa, tb;
        if (wi.z > fabsf(wo.z)) { sa = so; tb = si / fabsf(wi.z); }        // abs(Bool) quirk, Q18
        else { sa = si; tb = so / fabsf(wo.z); }
        return l.r * (1.0f / TR_PI) * (l.ax + l.ay * max_cos * sa * tb);
    }
    return f3s(0.0f);      // delta lobes
}
__device__ __forceinline__ float lobe_pdf(const Lobe& l, float3 wo, float3 wi) {
    if (l.kind == LK_FRESNEL_SPEC) return 0.0f;
    if (l.kind == LK_MICRO_REFL) {
        if (!same_hemi(wo, wi)) return 0.0f;
        float3 wh = normalize3(wo + wi);
        return tr_pdf(l, wo, wh) / dot3(4.0f * wo, wh);
    }
    if (l.kind == LK_MICRO_TRANS) {                    // microfacet.jl:322-337
        if (same_hemi(wo, wi)) return 0.0f;
        const float eta = wo.z > 0.0f ? (l.eta_b / l.eta_a) : (l.eta_a / l.eta_b);
        const float3 wh = normalize3(wo + wi * eta);
        const float d_o = dot3(wo, wh), d_i = dot3(wi, wh);
        if (d_o * d_i > 0.0f) return 0.0f;
        const float denom = d_o + eta * d_i;
        return tr_pdf(l, wo, wh) * fabsf(d_i * (eta * eta) / (denom * denom));
    }
    return same_hemi(wo, wi) ? fabsf(wi.z) * (1.0f / TR_PI) : 0.0f;
}
struct LobeSample { float3 wi, f; float pdf; int sampled_type; };
__device__ __forceinline__ LobeSample lobe_sample(const Lobe& l, float3 wo, float u0, float u1) {
    LobeSample s; s.wi = f3s(0.0f); s.f = f3s(0.0f); s.pdf = 0.0f; s.sampled_type = -1;
    if (l.kind == LK_SPEC_REFL) {
        s.wi = f3(-wo.x, -wo.y, wo.z); s.pdf = 1.0f;
        s.f = (lobe_fresnel(l, s.wi.z) * l.r) / fabsf(s.wi.z);
    } else if (l.kind == LK_SPEC_TRANS) {
        bool entering = wo.z > 0.0f;
        float ei = entering ? l.eta_a : l.eta_b, et = entering ? l.eta_b : l.eta_a;
        float3 wi;
        if (!refract(wo, face_forward(f3(0.0f, 0.0f, 1.0f), wo), ei / et, wi)) return s;
        s.wi = wi; s.pdf = 1.0f;
        float3 ft = l.t * (f3s(1.0f) - f3s(fresnel_dielectric(wi.z, l.eta_a, l.eta_b)));
        s.f = ft / fabsf(wi.z);
    } else if (l.kind == LK_FRESNEL_SPEC) {
        float fd = fresnel_dielectric(wo.z, l.eta_a, l.eta_b);
        if (u0 < fd) {
            s.wi = f3(-wo.x, -wo.y, wo.z); s.sampled_type = LB_SPECULAR | LB_REFLECTION; s.pdf = fd;
            s.f = (fd * l.r) / fabsf(s.wi.z);
            return s;
        }
        float ei, et;
        if (wo.z > 0.0f) { ei = l.eta_a; et = l.eta_b; } else { ei = l.eta_b; et = l.eta_a; }
        float3 wi;
        if (!refract(wo, face_forward(f3(0.0f, 0.0f, 1.0f), wo), ei / et, wi)) { s.wi = wi; s.pdf = fd; return s; }
        float pdf = 1.0f - fd;
        s.wi = wi; s.pdf = pdf; s.f = (l.t * pdf) / fabsf(wi.z);
        s.sampled_type = LB_SPECULAR | LB_TRANSMISSION;
    } else if (l.kind == LK_MICRO_REFL) {
        if (wo.z == 0.0f) return s;
        float3 wh = tr_sample_wh(l, wo, u0, u1);
        if (dot3(wo, wh) < 0.0f) return s;
        float3 wi = -wo + (2.0f * dot3(wo, wh)) * wh;
        if (!same_hemi(wo, wi)) return s;
        s.wi = wi;
        s.pdf = lobe_pdf(l, wo, wh);          // Q27: BxDF-level pdf evaluated with wh in the wi slot
        s.f = lobe_f(l, wo, wi);
    } else if (l.kind == LK_MICRO_TRANS) {             // microfacet.jl:307-320
        if (wo.z == 0.0f) return s;
        float3 wh = tr_sample_wh(l, wo, u0, u1);
        if (dot3(wo, wh) < 0.0f) return s;
        const float eta = wo.z > 0.0f ? (l.eta_b / l.eta_a) : (l.eta_a / l.eta_b);
        float3 wi;
        if (!refract(wo, wh, eta, wi)) return s;
        s.wi = wi; s.pdf = lobe_pdf(l, wo, wi); s.f = lobe_f(l, wo, wi);
    } else {
        float3 wi = cosine_hemisphere(u0, u1);
        if (wo.z < 0.0f) wi = f3(wi.x, wi.y, -wi.z);
        s.wi = wi; s.pdf = lobe_pdf(l, wo, wi); s.f = lobe_f(l, wo, wi);
    }
    return s;
}

// ------------------------------------------------------------------ BSDF-level f / sample_f, materials/bsdf.jl:79-175
__device__ __forceinline__ float3 bsdf_f(const LobeSet& s, const Frame& fr, float3 wo_w, float3 wi_w, uint32_t flags) {
    float3 wo = to_local(fr, wo_w);
    if (wo.z == 0.0f) return f3s(0.0f);
    float3 wi = to_local(fr, wi_w);
    bool reflect = dot3(wi_w, fr.ng) * dot3(wo_w, fr.ng) > 0.0f;
    float3 out = f3s(0.0f);
    for (int i = 0; i < s.n; ++i) {
        const Lobe& l = s.l[i];
        if (lobe_matches(l, flags) && ((reflect && (l.type & LB_REFLECTION)) || (!reflect && (l.type & LB_TRANSMISSION))))
            out = out + lobe_f(l, wo, wi);
    }
    return out;
}
struct BSDFSample { float3 wi, f; float pdf; uint32_t type; };
__device__ __forceinline__ BSDFSample bsdf_sample(const LobeSet& s, const Frame& fr, float3 wo_w, float u0, float u1, uint32_t type) {
    BSDFSample none; none.wi = f3s(0.0f); none.f = f3s(0.0f); none.pdf = 0.0f; none.type = 0;
    int mc = num_components(s, type);
    if (mc == 0) return none;
    int comp = (int)ceilf(u0 * (float)mc);
    comp = min(max(1, comp), mc);
    int count = comp, chosen = 0;
    comp -= 1;
    for (int i = 0; i < s.n; ++i) {
        if (lobe_matches(s.l[i], type)) {
            if (count == 1) { chosen = i; break; }
            count -= 1;
        }
    }
    const Lobe& bx = s.l[chosen];
    float ur0 = jl_min1(u0 * (float)mc - (float)comp);
    float3 wo = to_local(fr, wo_w);
    if (wo.z == 0.0f) return none;
    LobeSample ls = lobe_sample(bx, wo, ur0, u1);
    uint32_t sampled = ls.sampled_type >= 0 ? (uint32_t)ls.sampled_type : bx.type;
    if (ls.pdf == 0.0f) return none;
    float pdf = ls.pdf;
    float3 f = ls.f;
    float3 wi_w = to_world(fr, ls.wi);
    bool spec = (bx.type & LB_SPECULAR) != 0;
    if (!spec && mc > 1) {
        for (int i = 0; i < s.n; ++i)
            if (i != chosen && lobe_matches(s.l[i], type)) pdf += lobe_pdf(s.l[i], wo, ls.wi);
    }
    if (mc > 1) pdf /= (float)mc;
    if (!spec) {
        bool reflect = dot3(wi_w, fr.ng) * dot3(wo_w, fr.ng) > 0.0f;
        f = f3s(0.0f);
        for (int i = 0; i < s.n; ++i) {
            const Lobe& l = s.l[i];
            if (lobe_matches(l, type) && ((reflect && (l.type & LB_REFLECTION)) || (!reflect && (l.type & LB_TRANSMISSION))))
                f = f + lobe_f(l, wo, ls.wi);
        }
    }
    BSDFSample r; r.wi = wi_w; r.f = f; r.pdf = pdf; r.type = sampled;
    return r;
}

// ------------------------------------------------------------------ lights, lights/point.jl + spot.jl
__device__ __forceinline__ float spot_falloff(const DeviceLight& l, float3 w) {
    float3 wl = normalize3(xform_vector(l.inv_m, w));
    float c = wl.z;
    if (c < l.cos_total) return 0.0f;
    if (c >= l.cos_falloff) return 1.0f;
    float d = (c - l.cos_total) / (l.cos_falloff - l.cos_total);
    return pow4f(d);
}
// sample_li: radiance arriving at p, unit direction wi towards the light, light position
__device__ __forceinline__ float3 sample_li(const DeviceLight& l, float3 p, float3& wi, float3& lpos) {
    lpos = f3(l.pos[0], l.pos[1], l.pos[2]);
    float3 dd = lpos - p;
    wi = normalize3(dd);
    float d2 = dot3(dd, dd);
    float3 I = f3(l.I[0], l.I[1], l.I[2]);
    if (l.kind == TRACE_LIGHT_POINT) return I / d2;
    return (I * spot_falloff(l, -wi)) / d2;
}
// DirectionalLight.sample_li (lights/directional.jl:39-47): wi = direction, Li = I, the shadow ray ends at
// p + direction * 2 * world_radius (world_radius stays 0 unless the user ran preprocess!)
__device__ __forceinline__ float3 sample_li_any(const DeviceLight& l, float3 p, float3& wi, float3& lpos) {
    if (l.kind != TRACE_LIGHT_DIRECTIONAL) return sample_li(l, p, wi, lpos);
    wi = f3(l.pos[0], l.pos[1], l.pos[2]);
    lpos = p + wi * (2.0f * l.cos_total);
    return f3(l.I[0], l.I[1], l.I[2]);
}
__device__ __forceinline__ float3 light_power(const DeviceLight& l) {
    float3 I = f3(l.I[0], l.I[1], l.I[2]);
    if (l.kind == TRACE_LIGHT_POINT) return (4.0f * TR_PI) * I;
    if (l.kind == TRACE_LIGHT_DIRECTIONAL) return (I * TR_PI) * (l.cos_total * l.cos_total);
    return ((I * 2.0f) * TR_PI) * (1.0f - 0.5f * (l.cos_falloff + l.cos_total));
}

// ------------------------------------------------------------------ camera, camera/perspective.jl:85-114
__device__ __forceinline__ void generate_camera_ray(const DeviceCamera& c, float fx, float fy, float lu, float lv,
                                                    float3& o, float3& d) {
    float3 pc = xform_point(c.r2c, f3(fx, fy, 0.0f));
    o = f3s(0.0f);
    d = normalize3(pc);
    if (c.lens_radius > 0.0f) {
        float2 pl = concentric_disk(lu, lv);
        pl.x = c.lens_radius * pl.x; pl.y = c.lens_radius * pl.y;
        float t = c.focal_distance / d.z;
        float3 pf = o + d * t;
        o = f3(pl.x, pl.y, 0.0f);
        d = normalize3(pf - o);
    }
    o = xform_point(c.c2w, o);
    d = normalize3(xform_vector(c.c2w, d));
}

// ------------------------------------------------------------------ Halton, sampler/sampling.jl:43-76
// PRIMES of the reference (sampler/primes.jl): the 1023 odd primes 3 .. 8161, i.e. Halton dimension k >= 1 uses the
// (k+1)-th prime.  Generated at compile time (sieve), not transcribed.
struct PrimeTable {
    int v[1023];
    constexpr PrimeTable() : v{} {
        bool composite[8200] = {};
        int n = 0;
        for (int i = 2; i < 8200 && n < 1023; ++i) {
            if (composite[i]) continue;
            if (i > 2) v[n++] = i;
            for (int j = i * i; j < 8200; j += i) composite[j] = true;
        }
    }
};
__constant__ PrimeTable c_primes = PrimeTable();
#define TR_MAX_HALTON_DIM 1023
__device__ __forceinline__ float radical_inverse(int base_index, unsigned long long a) {
    if (base_index == 0) return (float)((double)__brevll(a) * 5.4210108624275222e-20);
    const unsigned long long base = (unsigned long long)c_primes.v[min(base_index, TR_MAX_HALTON_DIM) - 1];
    const float inv_base = 1.0f / (float)base;
    unsigned long long reversed = 0;
    float inv_base_n = 1.0f;
    while (a > 0) {
        // floor(a / base) in Float64 as the reference does; a < 2^53 here so it equals the integer quotient
        unsigned long long next = (unsigned long long)floor((double)a / (double)base);
        unsigned long long digit = a - next * base;
        reversed = reversed * base + digit;
        inv_base_n *= inv_base;
        a = next;
    }
    return fminf((float)reversed * inv_base_n, 1.0f);
}
