// ref_scene.cpp — CPU ORACLE (test infrastructure only): closest-hit / any-hit traversal and the two shape tests.
// Follows src/accel/bvh.jl:212-299, src/bounds.jl:169-200, src/ray.jl:25-29, src/shapes/triangle_mesh.jl:65-273,
// src/shapes/sphere.jl:39-191, src/primitive.jl:12-26, src/surface_interaction.jl:51-88,154-181.
#include <thread>

#include "ref_internal.hpp"

namespace ref {

// ---- bounds.jl:180-200. slab == 0: literal (line 191 keeps the LARGER y far bound, Q26); slab == 1: standard.
bool slab_test(const float* bmin, const float* bmax, const Ray& r, V3 inv, const int neg[3], int slab) {
    float tx_min = ((neg[0] ? bmax[0] : bmin[0]) - r.o.x) * inv.x;
    float tx_max = ((neg[0] ? bmin[0] : bmax[0]) - r.o.x) * inv.x;
    float ty_min = ((neg[1] ? bmax[1] : bmin[1]) - r.o.y) * inv.y;
    float ty_max = ((neg[1] ? bmin[1] : bmax[1]) - r.o.y) * inv.y;
    if (tx_min > ty_max || ty_min > tx_max) return false;
    if (ty_min > tx_min) tx_min = ty_min;
    if (slab == 0) { if (ty_max > tx_max) tx_max = ty_max; }
    else           { if (ty_max < tx_max) tx_max = ty_max; }
    float tz_min = ((neg[2] ? bmax[2] : bmin[2]) - r.o.z) * inv.z;
    float tz_max = ((neg[2] ? bmin[2] : bmax[2]) - r.o.z) * inv.z;
    if (tx_min > tz_max || tz_min > tx_max) return false;
    if (tz_min > tx_min) tx_min = tz_min;
    if (tz_max < tx_max) tx_max = tz_max;
    return tx_min < r.t_max && tx_max > 0.0f;
}

// ---- triangle_mesh.jl:187-218 / 245-273. Returns hit; fills t and barycentrics.
static bool triangle_test(const Tri& tri, const Ray& ray, float& t_hit, float bary[3]) {
    const V3 &p0 = tri.p[0], &p1 = tri.p[1], &p2 = tri.p[2];
    V3 dg = cross(p2 - p0, p1 - p0);                         // is_degenerate :65-68
    if (dot(dg, dg) == 0.0f) return false;
    // _to_ray_coordinate_space :99-123
    float ax = fabsf(ray.d.x), ay = fabsf(ray.d.y), az = fabsf(ray.d.z);
    int kz = 0; float am = ax;
    if (ay > am) { kz = 1; am = ay; }
    if (az > am) { kz = 2; am = az; }
    int kx = kz + 1; if (kx == 3) kx = 0;
    int ky = kx + 1; if (ky == 3) ky = 0;
    float dx = ray.d[kx], dy = ray.d[ky], dz = ray.d[kz];
    float denom = 1.0f / dz;
    float sx = -dx * denom, sy = -dy * denom, sz = denom;
    float X[3], Y[3], Z[3];
    for (int i = 0; i < 3; ++i) {
        V3 q = tri.p[i] - ray.o;
        float qz = tri.p[i][kz] - ray.o[kz];
        X[i] = q[kx] + sx * qz;
        Y[i] = q[ky] + sy * qz;
        Z[i] = q[kz] + 0.0f;
    }
    // _edge_function :85-91
    float e0 = X[1] * Y[2] - Y[1] * X[2];
    float e1 = X[2] * Y[0] - Y[2] * X[0];
    float e2 = X[0] * Y[1] - Y[0] * X[1];
    if (e0 == 0.0f && e1 == 0.0f && e2 == 0.0f) {             // iszero(edges): ALL zero -> Float64 fallback :195-197
        e0 = (float)((double)X[1] * (double)Y[2] - (double)Y[1] * (double)X[2]);
        e1 = (float)((double)X[2] * (double)Y[0] - (double)Y[2] * (double)X[0]);
        e2 = (float)((double)X[0] * (double)Y[1] - (double)Y[0] * (double)X[1]);
    }
    if ((e0 < 0.0f || e1 < 0.0f || e2 < 0.0f) && (e0 > 0.0f || e1 > 0.0f || e2 > 0.0f)) return false;
    float det = (e0 + e1) + e2;
    if (det == 0.0f) return false;                            // det ≈ 0 (isapprox to zero == exact zero)
    float ts = ((e0 * Z[0]) * sz + (e1 * Z[1]) * sz) + (e2 * Z[2]) * sz;
    if (det < 0.0f && (ts >= 0.0f || ts < ray.t_max * det)) return false;
    if (det > 0.0f && (ts <= 0.0f || ts > ray.t_max * det)) return false;
    float inv_det = 1.0f / det;
    bary[0] = e0 * inv_det; bary[1] = e1 * inv_det; bary[2] = e2 * inv_det;
    t_hit = ts * inv_det;
    return true;
}

// ---- sphere.jl:39-75,125-191
struct SphereHit { float t; V3 p; float phi; };

static V3 refine_intersection(V3 p, float radius) {           // :56-60
    float f = radius / norm(V3(0.0f) - p);
    p = p * f;
    if (p.x == 0.0f && p.y == 0.0f) p = V3(1e-6f * radius, p.y, p.z);
    return p;
}
static float compute_phi(V3 p) {                               // :71-75
    float phi = atan2f(p.y, p.x);
    if (phi < 0.0f) phi += 2.0f * PI_F;
    return phi;
}
static bool test_clipping(const trace_sphere& s, V3 p, float phi) {   // :65-69
    return (s.z_min > -s.radius && p.z < s.z_min) || (s.z_max < s.radius && p.z > s.z_max) || phi > s.phi_max;
}
static bool sphere_test(const trace_sphere& s, const Ray& ray, SphereHit& h) {
    V3 o = xf_point(s.inv_m, ray.o);                           // world_to_object(ray), transformations.jl:144
    V3 d = xf_vector(s.inv_m, ray.d);
    float nd = norm(d), no = norm(o);
    float a = nd * nd;
    float b = dot(2.0f * o, d);
    float c = no * no - s.radius * s.radius;
    float disc = b * b - (4.0f * a) * c;                       // solve_quadratic :39-54
    if (disc < 0.0f) return false;
    float rd = sqrtf(disc);
    float q = -0.5f * (b + (b < 0.0f ? -rd : rd));
    float t0 = q / a, t1 = c / q;
    if (t0 > t1) { float tmp = t0; t0 = t1; t1 = tmp; }
    if (t0 > ray.t_max || t1 < 0.0f) return false;
    if (t0 < 0.0f) t0 = t1;                                    // no t_max re-check (Q12)
    h.t = t0;
    h.p = refine_intersection(o + d * t0, s.radius);
    h.phi = compute_phi(h.p);
    if (test_clipping(s, h.p, h.phi)) {
        h.t = t1;
        h.p = refine_intersection(o + d * t1, s.radius);
        h.phi = compute_phi(h.p);
        if (test_clipping(s, h.p, h.phi)) return false;
    }
    return true;
}

static inline void prepare_ray(Ray& ray, V3& inv, int neg[3]) {
    // check_direction! (ray.jl:25-29): only -0.0 becomes +0.0;  inv_dir, is_dir_negative (bvh.jl:217-219)
    if (ray.d.x == 0.0f) ray.d.x = 0.0f;
    if (ray.d.y == 0.0f) ray.d.y = 0.0f;
    if (ray.d.z == 0.0f) ray.d.z = 0.0f;
    inv = V3(1.0f / ray.d.x, 1.0f / ray.d.y, 1.0f / ray.d.z);
    neg[0] = ray.d.x < 0.0f; neg[1] = ray.d.y < 0.0f; neg[2] = ray.d.z < 0.0f;
}

bool intersect_closest(const Scene& s, Ray& ray, Hit& hit, int slab, Counters* cnt) {
    hit = Hit();
    if (s.nodes.empty()) return false;
    V3 inv; int neg[3];
    prepare_ray(ray, inv, neg);
    uint32_t stack[256];
    int to_visit = 0;
    uint32_t cur = 0;
    for (;;) {
        const trace_bvh_node& ln = s.nodes[cur];
        if (cnt) cnt->nodes++;
        if (slab_test(ln.bmin, ln.bmax, ray, inv, neg, slab)) {
            uint32_t n = ln.meta & 0x3FFFFFFFu;
            if ((ln.meta >> 30) == 3u && n > 0) {
                for (uint32_t i = 0; i < n; ++i) {
                    uint32_t pi = ln.offset + i;
                    const trace_prim& pr = s.prims[pi];
                    if (cnt) cnt->prims++;
                    if (pr.kind == TRACE_PRIM_TRIANGLE) {
                        float t, b[3];
                        if (triangle_test(s.tris[pr.index], ray, t, b)) {
                            ray.t_max = t;                      // primitive.jl:16
                            hit.hit = true; hit.prim = (int32_t)pi; hit.t = t;
                            hit.b[0] = b[0]; hit.b[1] = b[1]; hit.b[2] = b[2];
                        }
                    } else {
                        SphereHit sh;
                        if (sphere_test(s.spheres[pr.index], ray, sh)) {
                            ray.t_max = sh.t;
                            hit.hit = true; hit.prim = (int32_t)pi; hit.t = sh.t;
                            hit.b[0] = hit.b[1] = hit.b[2] = 0.0f;
                        }
                    }
                }
                if (to_visit == 0) break;
                cur = stack[--to_visit];
            } else {
                uint32_t axis = ln.meta >> 30;
                if (axis > 2) axis = 0;   // zero-primitive leaf: unreachable in practice (Q17)
                if (to_visit >= 255) return hit.hit;
                if (neg[axis]) { stack[to_visit++] = cur + 1; cur = ln.offset; }
                else           { stack[to_visit++] = ln.offset; cur = cur + 1; }
                if (cnt && (uint64_t)to_visit > cnt->max_stack) cnt->max_stack = to_visit;
            }
        } else {
            if (to_visit == 0) break;
            cur = stack[--to_visit];
        }
    }
    return hit.hit;
}

bool intersect_any(const Scene& s, Ray& ray, int slab, Counters* cnt) {
    if (s.nodes.empty()) return false;
    V3 inv; int neg[3];
    prepare_ray(ray, inv, neg);
    uint32_t stack[256];
    int to_visit = 0;
    uint32_t cur = 0;
    for (;;) {
        const trace_bvh_node& ln = s.nodes[cur];
        if (cnt) cnt->nodes++;
        if (slab_test(ln.bmin, ln.bmax, ray, inv, neg, slab)) {
            uint32_t n = ln.meta & 0x3FFFFFFFu;
            if ((ln.meta >> 30) == 3u && n > 0) {
                for (uint32_t i = 0; i < n; ++i) {
                    const trace_prim& pr = s.prims[ln.offset + i];
                    if (cnt) cnt->prims++;
                    if (pr.kind == TRACE_PRIM_TRIANGLE) {
                        float t, b[3];
                        if (triangle_test(s.tris[pr.index], ray, t, b)) return true;
                    } else {
                        SphereHit sh;
                        if (sphere_test(s.spheres[pr.index], ray, sh)) return true;
                    }
                }
                if (to_visit == 0) break;
                cur = stack[--to_visit];
            } else {
                uint32_t axis = ln.meta >> 30;
                if (axis > 2) axis = 0;
                if (to_visit >= 255) return false;
                if (neg[axis]) { stack[to_visit++] = cur + 1; cur = ln.offset; }
                else           { stack[to_visit++] = ln.offset; cur = cur + 1; }
            }
        } else {
            if (to_visit == 0) break;
            cur = stack[--to_visit];
        }
    }
    return false;
}

// ---- hit record of the winning candidate.
void build_interaction(const Scene& s, const Ray& ray, const Hit& hit, SurfaceInteraction& si) {
    const trace_prim& pr = s.prims[hit.prim];
    si.prim = hit.prim;
    si.material = pr.material;
    if (pr.kind == TRACE_PRIM_TRIANGLE) {
        // triangle_mesh.jl:220-242, 125-141, 160-185; surface_interaction.jl:51-88
        const Tri& tr = s.tris[pr.index];
        const V3 &p0 = tr.p[0], &p1 = tr.p[1], &p2 = tr.p[2];
        const float uv[3][2] = {{0.0f, 0.0f}, {1.0f, 0.0f}, {1.0f, 1.0f}};        // uvs(t) default :79-83
        float duv13[2] = {uv[0][0] - uv[2][0], uv[0][1] - uv[2][1]};
        float duv23[2] = {uv[1][0] - uv[2][0], uv[1][1] - uv[2][1]};
        V3 dp13 = p0 - p2, dp23 = p1 - p2;
        float det = duv13[0] * duv23[1] - duv13[1] * duv23[0];
        float inv_det = 1.0f / det;                                               // det == 1 for the default uv
        V3 dpdu = (duv23[1] * dp13 - duv13[1] * dp23) * inv_det;
        V3 dpdv = ((-duv23[0]) * dp13 + duv13[0] * dp23) * inv_det;
        (void)dpdv;
        si.p = (hit.b[0] * p0 + hit.b[1] * p1) + hit.b[2] * p2;                   // sum_mul, Trace.jl:98
        si.u = (hit.b[0] * uv[0][0] + hit.b[1] * uv[1][0]) + hit.b[2] * uv[2][0];
        si.v = (hit.b[0] * uv[0][1] + hit.b[1] * uv[1][1]) + hit.b[2] * uv[2][1];
        si.wo = -ray.d;
        V3 ng = normalize(cross(dp13, dp23));                                     // :230
        V3 ns = ng;
        si.sh_dpdu = dpdu;
        if (tr.has_normals) {                                                     // _init_triangle_shading_geometry!
            V3 ns0 = normalize((hit.b[0] * tr.n[0] + hit.b[1] * tr.n[1]) + hit.b[2] * tr.n[2]);
            V3 ss = normalize(dpdu);
            V3 ts = cross(ns0, ss);
            if (dot(ts, ts) > 0.0f) { ts = normalize(ts); ss = cross(ts, ns0); }
            else { V3 a, b2; coordinate_system(ns0, a, b2); ss = a; ts = b2; }
            ns = normalize(cross(ss, ts));                                        // set_shading_geometry! :74
            if (tr.flip) ns = ns * -1.0f;
            ng = face_forward(ng, ns);                                            // :78-79 and triangle_mesh.jl:234-237
            si.sh_dpdu = ss;
        } else if (tr.flip) {
            ng = -ng; ns = ng;
        }
        si.ng = ng; si.ns = ns;
    } else {
        // sphere.jl:150-163, 88-93; surface_interaction.jl:51-68, 154-181
        const trace_sphere& sp = s.spheres[pr.index];
        Ray r2 = ray; r2.t_max = INF_F;
        SphereHit sh;
        sphere_test(sp, r2, sh);
        V3 hp = sh.p;
        si.u = sh.phi / sp.phi_max;
        float theta = acosf(jl_clamp(hp.z / sp.radius, -1.0f, 1.0f));
        si.v = (theta - sp.theta_min) / (sp.theta_max - sp.theta_min);
        float z_radius = sqrtf(hp.x * hp.x + hp.y * hp.y);                        // precompute_ϕ :77-83
        float inv_zr = 1.0f / z_radius;
        float cos_phi = hp.x * inv_zr, sin_phi = hp.y * inv_zr;
        V3 dpdu(-sp.phi_max * hp.y, sp.phi_max * hp.x, 0.0f);
        V3 dpdv = (sp.theta_max - sp.theta_min) * V3(hp.z * cos_phi, hp.z * sin_phi, -sp.radius * sinf(theta));
        V3 n = normalize(cross(dpdu, dpdv));
        if (sp.flip) n = n * -1.0f;
        si.p = xf_point(sp.m, hp);
        si.wo = normalize(xf_vector(sp.m, -ray.d));
        si.ng = normalize(xf_normal(sp.inv_m, n));
        si.ns = si.ng;
        si.sh_dpdu = xf_vector(sp.m, dpdu);
    }
}

}  // namespace ref

using namespace ref;

extern "C" ref_scene* ref_scene_create(const trace_scene_desc* d) {
    ref_scene* rs = new ref_scene();
    Scene& s = rs->s;
    s.nodes.assign(d->nodes, d->nodes + d->n_nodes);
    s.prims.assign(d->prims, d->prims + d->n_prims);
    s.tris.resize(d->n_tris);
    for (int64_t i = 0; i < d->n_tris; ++i) {
        Tri& t = s.tris[i];
        const float* v = d->tri_vertices + 9 * i;
        for (int k = 0; k < 3; ++k) t.p[k] = V3(v[3 * k], v[3 * k + 1], v[3 * k + 2]);
        uint8_t fl = d->tri_flags ? d->tri_flags[i] : 0;
        t.flip = (fl & TRACE_TRI_FLIP) != 0;
        t.has_normals = d->tri_normals != nullptr && (fl & TRACE_TRI_HAS_NORMALS) != 0;
        if (t.has_normals) {
            const float* nn = d->tri_normals + 9 * i;
            for (int k = 0; k < 3; ++k) t.n[k] = V3(nn[3 * k], nn[3 * k + 1], nn[3 * k + 2]);
        }
    }
    if (d->n_spheres) s.spheres.assign(d->spheres, d->spheres + d->n_spheres);
    if (d->n_materials) s.materials.assign(d->materials, d->materials + d->n_materials);
    if (d->n_lights) s.lights.assign(d->lights, d->lights + d->n_lights);
    return rs;
}
extern "C" void ref_scene_free(ref_scene* s) { delete s; }

template <class F>
static void parallel_for(int64_t n, int n_threads, F f) {
    if (n_threads <= 1 || n < 1024) { f(0, n, 0); return; }
    std::vector<std::thread> th;
    int64_t chunk = (n + n_threads - 1) / n_threads;
    for (int t = 0; t < n_threads; ++t) {
        int64_t a = t * chunk, b = std::min(n, a + chunk);
        if (a >= b) break;
        th.emplace_back([=] { f(a, b, t); });
    }
    for (auto& x : th) x.join();
}

extern "C" int ref_intersect(const ref_scene* rs, const float* o, const float* d, float* tmax, int64_t n,
                             uint32_t* prim_out, float* b0b1, int slab, uint64_t* counters, int n_threads) {
    const Scene& s = rs->s;
    std::vector<Counters> cs(std::max(1, n_threads));
    parallel_for(n, n_threads, [&](int64_t a, int64_t b, int tid) {
        for (int64_t i = a; i < b; ++i) {
            Ray r; r.o = V3(o[3 * i], o[3 * i + 1], o[3 * i + 2]); r.d = V3(d[3 * i], d[3 * i + 1], d[3 * i + 2]);
            r.t_max = tmax[i]; r.time = 0.0f;
            Hit h;
            intersect_closest(s, r, h, slab, counters ? &cs[tid] : nullptr);
            if (h.hit) {
                tmax[i] = r.t_max;
                prim_out[i] = s.prims[h.prim].original + 1;
                if (b0b1) { b0b1[2 * i] = h.b[0]; b0b1[2 * i + 1] = h.b[1]; }
            } else {
                prim_out[i] = 0;
                if (b0b1) { b0b1[2 * i] = 0.0f; b0b1[2 * i + 1] = 0.0f; }
            }
        }
    });
    if (counters) {
        counters[0] = counters[1] = counters[2] = 0;
        for (auto& c : cs) { counters[0] += c.nodes; counters[1] += c.prims; counters[2] = std::max<uint64_t>(counters[2], c.max_stack); }
    }
    return 0;
}

extern "C" int ref_occluded(const ref_scene* rs, const float* o, const float* d, const float* tmax, int64_t n,
                            uint8_t* out, int slab, uint64_t* counters, int n_threads) {
    const Scene& s = rs->s;
    std::vector<Counters> cs(std::max(1, n_threads));
    parallel_for(n, n_threads, [&](int64_t a, int64_t b, int tid) {
        for (int64_t i = a; i < b; ++i) {
            Ray r; r.o = V3(o[3 * i], o[3 * i + 1], o[3 * i + 2]); r.d = V3(d[3 * i], d[3 * i + 1], d[3 * i + 2]);
            r.t_max = tmax[i]; r.time = 0.0f;
            out[i] = intersect_any(s, r, slab, counters ? &cs[tid] : nullptr) ? 1 : 0;
        }
    });
    if (counters) {
        counters[0] = counters[1] = counters[2] = 0;
        for (auto& c : cs) { counters[0] += c.nodes; counters[1] += c.prims; }
    }
    return 0;
}

// prim_index < 0: through the BVH (intersect!(bvh, ray)); otherwise intersect(shape, ray) on that primitive alone
// (src/shapes/triangle_mesh.jl:187, src/shapes/sphere.jl:125), as the reference's shape-level tests call it.
extern "C" int ref_hit_record(const ref_scene* rs, const float* o, const float* d, float tmax, float* out) {
    return ref_prim_hit_record(rs, -1, o, d, tmax, out);
}
extern "C" int ref_prim_hit_record(const ref_scene* rs, int64_t prim_index, const float* o, const float* d, float tmax, float* out) {
    const Scene& s = rs->s;
    Ray r; r.o = V3(o[0], o[1], o[2]); r.d = V3(d[0], d[1], d[2]); r.t_max = tmax; r.time = 0.0f;
    Hit h;
    for (int i = 0; i < 24; ++i) out[i] = 0.0f;
    if (prim_index < 0) {
        if (!intersect_closest(s, r, h, 0, nullptr)) return 0;
    } else {
        const trace_prim& pr = s.prims[prim_index];
        if (pr.kind == TRACE_PRIM_TRIANGLE) {
            float t, b[3];
            if (!triangle_test(s.tris[pr.index], r, t, b)) return 0;
            h.hit = true; h.prim = (int32_t)prim_index; h.t = t; h.b[0] = b[0]; h.b[1] = b[1]; h.b[2] = b[2];
            r.t_max = t;
        } else {
            SphereHit sh;
            if (!sphere_test(s.spheres[pr.index], r, sh)) return 0;
            h.hit = true; h.prim = (int32_t)prim_index; h.t = sh.t;
            r.t_max = sh.t;
        }
    }
    SurfaceInteraction si;
    build_interaction(s, r, h, si);
    V3 ss = normalize(si.sh_dpdu);          // BSDF frame, materials/bsdf.jl:41-45
    V3 ts = cross(si.ns, ss);
    out[0] = 1.0f; out[1] = r.t_max;
    const V3 vs[6] = {si.p, si.ng, si.ns, ss, ts, si.wo};
    for (int k = 0; k < 6; ++k) { out[2 + 3 * k] = vs[k].x; out[3 + 3 * k] = vs[k].y; out[4 + 3 * k] = vs[k].z; }
    out[20] = si.u; out[21] = si.v;
    out[22] = (float)s.prims[h.prim].original; out[23] = (float)si.material;
    return 1;
}

// ref_hit_record over n rays (out: 24 floats per ray, a miss is all zeros)
extern "C" int ref_hit_record_batch(const ref_scene* rs, int64_t n, const float* o, const float* d, const float* tmax, float* out,
                                    int n_threads) {
    parallel_for(n, n_threads, [&](int64_t a, int64_t b, int) {
        for (int64_t i = a; i < b; ++i) ref_prim_hit_record(rs, -1, o + 3 * i, d + 3 * i, tmax ? tmax[i] : INF_F, out + 24 * i);
    });
    return 0;
}

extern "C" int ref_bounds_intersect(const float bmin[3], const float bmax[3], const float o[3], const float d[3],
                                    float tmax, float* t0o, float* t1o) {        // bounds.jl:151-167
    float t0 = 0.0f, t1 = tmax;
    for (int i = 0; i < 3; ++i) {
        float inv = 1.0f / d[i];
        float tn = (bmin[i] - o[i]) * inv, tf = (bmax[i] - o[i]) * inv;
        if (tn > tf) { float x = tn; tn = tf; tf = x; }
        t0 = tn > t0 ? tn : t0;
        t1 = tf < t1 ? tf : t1;
        if (t0 > t1) { *t0o = 0.0f; *t1o = 0.0f; return 0; }
    }
    *t0o = t0; *t1o = t1;
    return 1;
}
extern "C" int ref_bounds_intersect_p(const float bmin[3], const float bmax[3], const float o[3], const float d[3],
                                      float tmax, int slab) {
    Ray r; r.o = V3(o[0], o[1], o[2]); r.d = V3(d[0], d[1], d[2]); r.t_max = tmax; r.time = 0;
    V3 inv(1.0f / r.d.x, 1.0f / r.d.y, 1.0f / r.d.z);
    int neg[3] = {r.d.x < 0.0f, r.d.y < 0.0f, r.d.z < 0.0f};
    return slab_test(bmin, bmax, r, inv, neg, slab) ? 1 : 0;
}
