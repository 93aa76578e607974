/* trace_ref.h — C API of the CPU ORACLE (libtrace_ref.so).
 *
 * TEST INFRASTRUCTURE ONLY. This library is a CPU restatement of the reference's
 * (pxl-th/Trace.jl) algorithm for the ray-tracing hot path. Only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
 * load it. The product (libtrace_cuda.so and the trace.jl_b200 package) never does.
 *
 * Parity status: the reference is Julia and cannot run in this image (no julia
 * binary), so the oracle is pinned against the known-answer tests the reference's
 * own test suite holds (test/test_intersection.jl, test/test_materials.jl,
 * test/runtests.jl) and against the published 1024x1024 "shadows" PNG landmarks.
 * At the bit level the StaticArrays boundary (norm/normalize/mat*vec association
 * order) is "parity unpinned"; see DESIGN.md.
 *
 * It consumes the same POD scene format as the CUDA library (include/trace_cuda.h).
 */
#ifndef TRACE_REF_H
#define TRACE_REF_H
#include "../include/trace_cuda.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ref_scene ref_scene;
typedef struct ref_bvh ref_bvh;

/* BVHAccel constructor, literal (src/accel/bvh.jl:55-206) */
int     ref_bvh_build(const float* prim_bounds, int64_t n, int max_node_primitives, ref_bvh** out);
int64_t ref_bvh_num_nodes(const ref_bvh*);
int     ref_bvh_max_depth(const ref_bvh*);
int     ref_bvh_copy(const ref_bvh*, trace_bvh_node* nodes_out, uint32_t* prim_order_out);
void    ref_bvh_free(ref_bvh*);

ref_scene* ref_scene_create(const trace_scene_desc* desc);
void       ref_scene_free(ref_scene*);

/* intersect!(bvh, ray) / intersect_p(bvh, ray). slab: 0 literal (bounds.jl:180-200), 1 standard.
 * counters (may be NULL): [0] nodes visited, [1] primitives tested, [2] max stack depth. */
int ref_intersect(const ref_scene*, const float* o, const float* d, float* tmax_inout, int64_t n,
                  uint32_t* prim_out, float* b0b1_out, int slab, uint64_t* counters, int n_threads);
int ref_occluded(const ref_scene*, const float* o, const float* d, const float* tmax, int64_t n,
                 uint8_t* out, int slab, uint64_t* counters, int n_threads);
/* full hit record for one ray: out[24] = hit, t, p(3), ng(3), ns(3), ss(3), ts(3), wo(3), uv(2), prim_original, material */
int ref_hit_record(const ref_scene*, const float* o, const float* d, float tmax, float* out24);
/* same record from intersect(shape, ray) on one primitive of the BVH-ordered list, bypassing the BVH */
int ref_prim_hit_record(const ref_scene*, int64_t prim_index, const float* o, const float* d, float tmax, float* out24);

/* Whitted / SPPM renders. RNG: the reference draws rand(); the oracle substitutes the counter-based
 * generator specified in DESIGN.md so that a GPU render with the same seed is comparable per sample. */
int ref_render_whitted(const ref_scene*, const trace_camera*, const trace_film_desc*, int spp, int max_depth,
                       uint64_t seed, float* film_xyzw_inout, int n_threads, int64_t max_tiles,
                       uint64_t* ray_counters /* [0] closest-hit rays, [1] shadow rays; may be NULL */);
int ref_render_sppm(const ref_scene*, const trace_camera*, const trace_film_desc*, float r0, int max_depth,
                    int n_iterations, int64_t photons_per_iteration, uint64_t seed, float* rgb_out,
                    int n_threads, uint64_t* ray_counters);

/* ---- unit-level entry points for the reference's known-answer tests ---- */
int   ref_bounds_intersect(const float bmin[3], const float bmax[3], const float o[3], const float d[3],
                           float tmax, float* t0, float* t1);                       /* bounds.jl:151-167 */
int   ref_bounds_intersect_p(const float bmin[3], const float bmax[3], const float o[3], const float d[3],
                             float tmax, int slab);                                  /* bounds.jl:180-200 */
float ref_fresnel_dielectric(float cos_i, float eta_i, float eta_t);                /* reflection/bxdf.jl:74-95 */
/* sample_f of single BxDFs in the local frame; out = wi(3), pdf, f(3), sampled_type (or -1) */
int   ref_fresnel_specular_sample(const float r[3], const float t[3], float eta_a, float eta_b,
                                  const float wo[3], const float u[2], float out[8]);
int   ref_microfacet_reflection_sample(const float r[3], float ax, float ay, int fresnel_kind /*0 noop,1 dielectric*/,
                                       float eta_i, float eta_t, const float wo[3], const float u[2], float out[8]);
int   ref_microfacet_transmission_sample(const float t[3], float ax, float ay, float eta_a, float eta_b,
                                         const float wo[3], const float u[2], float out[8]);   /* microfacet.jl:307-320 */
float ref_lanczos(float px, float py, float rx, float ry, float tau);               /* filter.jl:3-23 */
float ref_radical_inverse(int64_t base_index, uint64_t a);                           /* sampler/sampling.jl:43-60 */
float ref_roughness_to_alpha(float r);                                               /* microfacet.jl:79-84 */
/* BSDF-level: builds the BSDF of `material` on a canonical frame (ns=ng=z, ss=x) and evaluates
 * f(wo,wi) / sample_f(wo,u,type). mode: 0 = Whitted lobes, 1 = SPPM lobes (allow_multiple_lobes). */
int   ref_bsdf_f(const trace_material*, int mode, const float wo[3], const float wi[3], int flags, float f_out[3]);
int   ref_bsdf_sample(const trace_material*, int mode, const float wo[3], const float u[2], int type,
                      float out[8] /* wi(3), f(3), pdf, sampled_type */);
/* the same over n inputs: q[i] = {material index into mats, mode, flags / type}; n_lobes[i] = the BSDF's lobe count */
int   ref_bsdf_f_batch(const trace_material* mats, int64_t n, const int32_t* q, const float* wo, const float* wi,
                       float* f_out /* n x 3 */, int32_t* n_lobes);
int   ref_bsdf_sample_batch(const trace_material* mats, int64_t n, const int32_t* q, const float* wo, const float* u,
                            float* out /* n x 8 */, int32_t* n_lobes);
/* ref_hit_record over n rays (tmax may be NULL: Inf); out is n x 24, all zeros for a miss */
int   ref_hit_record_batch(const ref_scene*, int64_t n, const float* o, const float* d, const float* tmax, float* out,
                           int n_threads);
/* add_sample! on a FilmTile (film.jl:134-164): splats into tile pixel arrays of size (ty1-ty0+1) x (tx1-tx0+1) */
int   ref_film_tile_add_sample(const trace_film_desc*, const int tile_bounds[4] /* x0,y0,x1,y1 */,
                               float px, float py, const float rgb[3], float* contrib_rgb, float* weight_sum);
/* counter-based RNG shared by spec with the CUDA library (DESIGN.md "RNG") */
float ref_rng(uint64_t seed, uint32_t a, uint32_t b, uint32_t c);

#ifdef __cplusplus
}
#endif
#endif
