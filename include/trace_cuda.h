/* trace_cuda.h — C ABI of libtrace_cuda.so, the B200 (sm_100a) backend for the
 * ray-tracing hot path of pxl-th/Trace.jl.
 *
 * The reference is pure Julia and has no FFI; the seams this ABI replaces are
 * ordinary Julia methods (citations are file:line under the reference tree):
 *
 *   trace_bvh_build            <- BVHAccel(primitives, max_node_primitives)   src/accel/bvh.jl:55-80 (+ _init :87-185, _unroll :187-206)
 *   trace_scene_upload         <- Scene(lights, aggregate)                    src/Trace.jl:176-187
 *   trace_scene_upload_mesh_device  (extension: a triangle scene built and packed on the GPU from device arrays)
 *   trace_scene_attach_mesh_device  (extension: such a mesh attached to the uploaded scene, rebuilt alone per frame)
 *   trace_scene_attach_meshes_device (extension: several such meshes, each rebuilt only when it changes)
 *   trace_intersect            <- intersect!(bvh|scene, ray)                  src/accel/bvh.jl:212-258, src/Trace.jl:189-191
 *   trace_occluded             <- intersect_p(bvh|scene, ray)                 src/accel/bvh.jl:260-299, src/Trace.jl:192-194
 *   trace_render_whitted       <- (i::SamplerIntegrator)(scene)               src/integrators/sampler.jl:12-56
 *   trace_render_sppm          <- (i::SPPMIntegrator)(scene)                  src/integrators/sppm.jl:132-173
 *   trace_sppm_* (stepwise)    <- the four per-iteration passes               src/integrators/sppm.jl:153-171
 *
 * Conventions: every function returns 0 on success and nonzero on failure
 * (trace_last_error gives the text); no exception crosses the ABI; all
 * pointer arguments are caller-owned and are not retained after the call
 * returns unless the name ends in _device (then they are device pointers on
 * the context's GPU); calls on one context must be serialised by the caller.
 * Indices are 0-based on this side of the ABI.
 */
#ifndef TRACE_CUDA_H
#define TRACE_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TRACE_ABI_VERSION 3

/* ---- BVH node, 32 bytes (LinearBVHLeaf / LinearBVHInterior, src/accel/bvh.jl:38-48) ----
 * interior: first child = self + 1, second child = `offset`; meta = split_axis << 30 (axis 0,1,2)
 * leaf:     primitives offset .. offset + n - 1 in the ordered primitive list; meta = 0xC0000000 | n
 */
#define TRACE_NODE_LEAF 0xC0000000u
typedef struct trace_bvh_node {
    float bmin[3];
    float bmax[3];
    uint32_t offset;
    uint32_t meta;
} trace_bvh_node;

/* ---- shapes ---- */
enum { TRACE_PRIM_TRIANGLE = 0, TRACE_PRIM_SPHERE = 1 };
enum { TRACE_TRI_FLIP = 1u,        /* reverse_orientation xor transform_swaps_handedness (src/shapes/Shape.jl:1-15) */
       TRACE_TRI_HAS_NORMALS = 2u  /* mesh.normals !== nothing (src/shapes/triangle_mesh.jl:9) */ };

/* Sphere (src/shapes/sphere.jl:1-25). Matrices are row-major 4x4: m = object_to_world.m,
 * inv_m = object_to_world.inv_m (so world_to_object.m == inv_m, src/transformations.jl:12). */
typedef struct trace_sphere {
    float m[16];
    float inv_m[16];
    float radius, z_min, z_max, theta_min, theta_max, phi_max;
    uint32_t flip;      /* reverse_orientation xor transform_swaps_handedness */
    uint32_t pad;
} trace_sphere;

/* One entry of the BVH-ordered primitive list (bvh.primitives, src/accel/bvh.jl:51,67,100-105). */
typedef struct trace_prim {
    uint32_t kind;      /* TRACE_PRIM_* */
    uint32_t index;     /* into tri_* arrays or spheres */
    uint32_t material;  /* into materials */
    uint32_t original;  /* index the caller wants reported back for this primitive */
} trace_prim;

/* ---- materials (src/materials/material.jl), constant textures only ---- */
enum { TRACE_MAT_MATTE = 0, TRACE_MAT_MIRROR = 1, TRACE_MAT_GLASS = 2, TRACE_MAT_PLASTIC = 3 };
typedef struct trace_material {
    uint32_t kind;
    float a[3];          /* Matte Kd | Mirror Kr | Glass Kr | Plastic Kd */
    float b[3];          /* Glass Kt | Plastic Ks */
    float eta;           /* Glass index */
    float rough_u;       /* Glass u_roughness | Plastic roughness | Matte sigma */
    float rough_v;       /* Glass v_roughness */
    uint32_t remap;      /* remap_roughness */
} trace_material;

/* ---- lights (src/lights/point.jl, spot.jl) ---- */
enum { TRACE_LIGHT_POINT = 0, TRACE_LIGHT_SPOT = 1,
       TRACE_LIGHT_DIRECTIONAL = 2 /* src/lights/directional.jl: position = normalised world direction, cos_total_width = world_radius */ };
typedef struct trace_light {
    uint32_t kind;
    float m[16];         /* light_to_world.m, row-major */
    float inv_m[16];     /* light_to_world.inv_m (== world_to_light.m) */
    float I[3];
    float position[3];   /* light_to_world(Point3f(0)) */
    float cos_total_width, cos_falloff_start;   /* spot only */
} trace_light;

typedef struct trace_scene_desc {
    int64_t n_nodes;      const trace_bvh_node* nodes;
    int64_t n_prims;      const trace_prim* prims;          /* BVH leaf order */
    int64_t n_tris;       const float* tri_vertices;        /* [n_tris][3][3], world space (TriangleMesh ctor transforms them, triangle_mesh.jl:23) */
                          const float* tri_normals;         /* [n_tris][3][3] or NULL */
                          const uint8_t* tri_flags;         /* [n_tris] TRACE_TRI_* */
    int64_t n_spheres;    const trace_sphere* spheres;
    int64_t n_materials;  const trace_material* materials;
    int64_t n_lights;     const trace_light* lights;
} trace_scene_desc;

/* ---- camera (src/camera/perspective.jl). The host builds the two matrices with the
 * reference's literal Transformation algebra (transformations.jl:20-22) and hands them over. ---- */
typedef struct trace_camera {
    float raster_to_camera[16];   /* .m, row-major */
    float camera_to_world[16];    /* .m, row-major */
    float lens_radius, focal_distance, shutter_open, shutter_close;
} trace_camera;

/* ---- film (src/film.jl:7-62). Pixel coordinates are 1-based like the reference's. ---- */
typedef struct trace_film_desc {
    int32_t crop_x0, crop_y0, crop_x1, crop_y1;   /* crop_bounds, inclusive, 1-based */
    float filter_radius[2];
    float filter_table[256];                        /* [y][x], 16x16 (film.jl:52-56) */
    float scale;
} trace_film_desc;

/* kernel classes of the per-class timing in trace_stats */
enum { TRACE_K_EXTEND = 0, TRACE_K_SHADOW = 1, TRACE_K_GENERATE = 2, TRACE_K_SHADE = 3, TRACE_K_SPLAT = 4,
       TRACE_K_GRID = 5 /* SPPM hash grid: bounds, count, scan, fill */, TRACE_K_DEPOSIT = 6, TRACE_K_UPDATE = 7,
       TRACE_K_COMM = 8 /* the library's NCCL collectives (film sum; visible-point all-gather, flux all-reduce) */,
       TRACE_K_COUNT = 9 };
typedef struct trace_stats {
    uint64_t rays_extend;        /* rays through closest-hit traversal */
    uint64_t rays_shadow;        /* rays through any-hit traversal */
    uint64_t nodes_visited;      /* only counted when option "count_nodes" is 1 or 2 */
    uint64_t prims_tested;
    uint64_t kernel_launches;    /* launches of this library's kernels since the last reset */
    double   ms_extend;          /* CUDA-event time in closest-hit kernels (option "time_kernels") */
    double   ms_shadow;
    double   ms_total;           /* CUDA-event time of the last render / query call, device side */
    uint64_t queue_overflows;    /* wavefront batches re-run because a ray queue overflowed */
    uint64_t sppm_deposits;
    uint64_t extend_launches;    /* closest-hit kernel launches timed into ms_extend */
    uint64_t shadow_launches;    /* any-hit kernel launches timed into ms_shadow */
    /* option "time_kernels": CUDA-event time and launch count per kernel class (TRACE_K_*); [0] and [1] repeat
     * ms_extend / ms_shadow */
    double   ms_kind[TRACE_K_COUNT];
    uint64_t launches_kind[TRACE_K_COUNT];
    uint64_t sppm_candidates;    /* visible points examined by photon deposits (16 B each, streamed) */
    uint64_t sppm_requests;      /* photon deposit requests (photon-surface hits at depth > 1) */
    uint64_t sppm_grid_items;    /* (visible point, grid cell) entries inserted */
    uint64_t primary_rays;       /* Whitted: camera rays traced ... */
    uint64_t primary_hits;       /* ... and how many of them hit something (the rest leave the scene after a few box tests) */
} trace_stats;

typedef struct trace_ctx trace_ctx;
typedef struct trace_bvh trace_bvh;

/* ---- host-side BVH build, no GPU needed (multi-threaded: TRACE_BVH_THREADS, default all cores; the tree does not depend on
 * the thread count).  Return codes: 0 ok, 1 bad argument, 2 out of memory, 3 / 4 node count out of range, 5 a primitive
 * bound is NaN (the reference's Int64(floor(NaN)) throws an InexactError there, src/accel/bvh.jl:118) ---- */
int     trace_bvh_build(const float* prim_bounds /* [n][6] = min xyz, max xyz */, int64_t n,
                        int max_node_primitives, trace_bvh** out);
/* opt-in: conventional binned SAH (primitive-count weighted, empty buckets, leaves up to max_node_primitives) in the same
 * node format.  Not the reference's tree: closest hits agree except for ties between equal t (SURVEY.md §8f.2). */
int     trace_bvh_build_sah(const float* prim_bounds, int64_t n, int max_node_primitives, trace_bvh** out);
/* opt-in: LBVH (Karras 2012 radix tree over 63-bit Morton codes of the centroids) built on GPU `device`, in the same
 * node format; the tree comes back as an ordinary host trace_bvh handle (trace_bvh_num_nodes / _copy / _free apply).
 * Not the reference's tree: closest hits agree except for ties between equal t.  max_node_primitives is clamped to
 * 1..255; a range of at most that many primitives is one leaf.  Synchronous; the caller's current device is restored;
 * TRACE_BVH_PROFILE=1 prints per-phase CUDA-event times to stderr.  Return codes as trace_bvh_build, plus 6: the tree
 * is deeper than the traversal stack (64 levels; builder "sah" handles such inputs), 7: CUDA error / no device (there
 * is no CPU fallback). */
int     trace_bvh_build_gpu(int device, const float* prim_bounds, int64_t n, int max_node_primitives, trace_bvh** out);
int64_t trace_bvh_num_nodes(const trace_bvh* bvh);
int64_t trace_bvh_num_prims(const trace_bvh* bvh);
int     trace_bvh_copy(const trace_bvh* bvh, trace_bvh_node* nodes_out, uint32_t* prim_order_out);
void    trace_bvh_free(trace_bvh* bvh);

/* ---- context ---- */
int         trace_abi_version(void);
int         trace_create(trace_ctx** out, int device, void* cuda_stream /* NULL: library-owned stream */);
void        trace_destroy(trace_ctx* ctx);
const char* trace_last_error(const trace_ctx* ctx);
/* options: "slab" 0 = literal reference slab test (bounds.jl:180-200), 1 = textbook slab (measured only: not
 *          hit-equivalent), 2 = guarded: literal AND a conservative interval test, hit-identical to 0 (default 2);
 *          "batch" camera samples in flight per Whitted render (default 2^26); "cap_percent" ray-queue capacity per
 *          bounce level in % of the batch (default 200; an overflowing batch is re-run in halves); "lanes" sub-batches
 *          of a Whitted render in flight concurrently on side streams (1..16, default 12); "deal" how tiles are dealt
 *          to those batches (g > 0: groups of g tiles, -r: r tile rows, 0: contiguous bands; default -2); "graph" 0/1
 *          replay the render as one CUDA graph (default 1; needs a non-default stream); "sppm_lanes" sub-ranges of
 *          each SPPM pass on concurrent streams (0..8, default 0 = one camera + one photon lane); "sppm_pipeline" SPPM
 *          iterations in flight (1..8, default 4): the camera pass and the photon tracing of later iterations run on
 *          their own streams and buffers while the serial chain grid -> deposits -> all-reduce -> update of the current
 *          one runs ("sppm_chain_priority" 0/1, default 1: that chain on a high-priority stream); "film_sum" how the
 *          whole film reaches rank 0 in film_mode 0: 0 ncclReduce (default), 1 ncclAllReduce, 2 reduce-scatter + gather of the
 *          chunks; "film_p2p" 0/1 (default 1): with a communicator of <= 8 ranks the film sum and the merge are one kernel
 *          over peer memory (the ranks' private films mapped into every process), "film_sum" then only names the NCCL
 *          fallback; "walk" traversal
 *          loop: 1 = pair nodes (default: one 64-byte fetch serves both children's box tests and the far child is
 *          pushed with its entry distance; same hits bit for bit), 0 = one node per step exactly as
 *          src/accel/bvh.jl:221-257; "leaf_wait" 0/4/8/16/32 warp-synchronous variant of loop 0 with batched leaf
 *          tests (measured slower, kept for the record); "film_mode" see trace_comm_init; "persist" 0/1
 *          persistent-warp traversal kernels (default 0); "count_nodes" 0/1/2 (2: closest hits count the
 *          "hit_tree" walk the default path runs, 1: the reference tree's walk); "time_kernels" 0/1 (per-launch CUDA
 *          events; with TRACE_CUDA_TIMELINE=<file> they are also dumped); "shadow_tree" 0/1 (default 1): any-hit queries
 *          (trace_occluded*, Whitted and SPPM shadow rays) walk the scene's shadow tree, an LBVH built on the device at
 *          upload, and check every occluder they find against the reference tree: the same answers bit for bit, 0 =
 *          walk the reference tree only (it applies with "slab" 2 and "walk" 1; a scene uploaded with 0 gets no shadow
 *          tree, which saves its 64 B per primitive); "hit_tree" 0/1 (default 1): closest-hit queries
 *          (trace_intersect*, Whitted and SPPM camera and photon rays) walk the shadow tree too and answer only when an
 *          exact check proves the reference walk returns the same primitive, else they run that walk: the same hits,
 *          t and barycentrics bit for bit, 0 = walk the reference tree only (it applies where "shadow_tree" does, and
 *          "shadow_tree" 0 turns it off as well); "rank"/"world" shard selection (Whitted: tiles
 *          k % world; SPPM: image rows and, through the photon range arguments, photons). */
int         trace_set_option(trace_ctx* ctx, const char* key, int64_t value);
int         trace_get_stats(trace_ctx* ctx, trace_stats* out);
int         trace_reset_stats(trace_ctx* ctx);
int         trace_synchronize(trace_ctx* ctx);

/* ---- multi-GPU: one trace_ctx per GPU (one per process, or one per thread of a process), scene uploaded to each.
 * The reference parallelises with Threads.@threads over 16x16 tiles (src/integrators/sampler.jl:24) and over photons
 * (src/integrators/sppm.jl:328) into SHARED film / pixel arrays; across GPUs the sharing becomes the two collectives of
 * SURVEY.md 8e, which the library runs itself on NCCL (bound at run time with dlopen; TRACE_NCCL_LIB overrides the
 * path).  Rank 0 creates an id, passes the TRACE_COMM_ID_BYTES bytes to the other ranks out of band, and all ranks
 * call trace_comm_init (collective: returns when all `world` ranks have joined).  Afterwards, on every rank,
 *   trace_render_whitted[_device] renders the rank's tiles (k % world == rank) and sums the films:
 *       option "film_mode" 0 (default): rank 0's film receives the whole image, other ranks' films are left untouched
 *                                       (their film pointer may be NULL in the host-buffer call);
 *       option "film_mode" 1: pixel i of the film (row-major) is delivered to rank i / ceil(n_pixels / world): every rank
 *                             adds its contiguous band to ITS film - threads of one process pass the same host film and
 *                             each GPU writes its band, processes each hold a band;
 *   trace_render_sppm shards camera paths by image rows and photons by index range, all-gathers the visible points and
 *       all-reduces (Phi, M) every iteration; every rank returns the complete image in rgb_out.
 * All ranks must make the same sequence of render calls with the same arguments. */
#define TRACE_COMM_ID_BYTES 128
int trace_comm_unique_id(void* id_out /* TRACE_COMM_ID_BYTES */);
int trace_comm_init(trace_ctx* ctx, const void* id, int rank, int world);
int trace_comm_destroy(trace_ctx* ctx);
int trace_comm_info(const trace_ctx* ctx, int* rank, int* world, int* nccl_version /* 0: no communicator */);

int trace_scene_upload(trace_ctx* ctx, const trace_scene_desc* scene);

/* ---- device mesh upload (extension: the reference has no counterpart).  A triangle-only scene whose per-triangle
 * arrays are already in device memory on the context's GPU: the GPU builds its tree (the LBVH of trace_bvh_build_gpu)
 * and writes every scene buffer; no array proportional to n_tris crosses to the host (the host reads the build's
 * status block and the root box).  The resulting device scene is bit for bit the one trace_scene_upload builds from
 *   nodes     = trace_bvh_build_gpu(device, B, n_tris, max_node_primitives), B[i] = Julia min / max (-0.0 < +0.0) of
 *               triangle i's three vertices (the refit's leaf rule);
 *   prims[k]  = {TRACE_PRIM_TRIANGLE, order[k], tri_materials[order[k]], order[k]}: `original` is the triangle index;
 *   the same triangle arrays (tri_normals NULL: zeros, TRACE_TRI_HAS_NORMALS cleared), no spheres, these materials
 *   and lights
 * - nodes, pair records, primitive records, normals and flags, shadow tree, scene_scale and counts alike.
 * Refused, before any scene buffer is written (the previous scene stays uploaded and usable): NaN in a vertex or a
 * normal, a material index >= n_materials, a tree deeper than 64 levels, n_tris >= 2^30, a NULL vertex array with
 * n_tris > 0, an unknown material or light kind.  n_tris == 0 uploads the empty scene, n_tris == 1 a single leaf.
 * The arrays are read on the context's stream: the caller orders the work that wrote them before this call.  Like
 * trace_scene_upload the call waits for all of the context's work, ends any SPPM session and is synchronous.  Its
 * scratch (the build's and the shadow tree's) lives in grow-only context buffers: a repeated upload of the same size
 * allocates nothing.  trace_scene_refit[_device] applies afterwards (the slot -> triangle map stays on the device).
 * *n_nodes_out (may be NULL) receives the node count.  TRACE_BVH_PROFILE=1 prints per-phase CUDA-event times. */
typedef struct trace_mesh_device_desc {
    int64_t n_tris;
    const void* tri_vertices;     /* device [n_tris][3][3] float32, world space */
    const void* tri_normals;      /* device [n_tris][3][3] float32, or NULL */
    const void* tri_flags;        /* device [n_tris] uint8 TRACE_TRI_*, or NULL (all 0) */
    const void* tri_materials;    /* device [n_tris] uint32 index into materials, or NULL (all 0) */
    int32_t max_node_primitives;  /* clamped to 1..255 as trace_bvh_build_gpu */
    int32_t pad;
    int64_t n_materials;  const trace_material* materials;   /* host */
    int64_t n_lights;     const trace_light* lights;         /* host */
} trace_mesh_device_desc;
int trace_scene_upload_mesh_device(trace_ctx* ctx, const trace_mesh_device_desc* mesh, int64_t* n_nodes_out);

/* ---- attach device meshes to the uploaded scene (extension: the reference has no counterpart).  The base is the scene
 * of the last trace_scene_upload or trace_scene_upload_mesh_device; a call composes it with the meshes of k slots,
 * each built from a descriptor (the same descriptor and checks as trace_scene_upload_mesh_device) or kept, while the
 * base stays resident.  The composed device scene is bit for bit the one trace_scene_upload builds from D:
 *   C(A, B)         the composition of two parts: a new root, interior, box = Julia min / max union of A's and B's
 *                   root boxes, first child A (node 1), second child B (offset 1 + NA); split axis = the k maximising
 *                   (B.min[k] + B.max[k]) - (A.min[k] + A.max[k]) in float32, ties to the lowest k, non-finite values
 *                   lose; then A's nodes (interior offsets + 1), then B's (interior offsets + 1 + NA, leaf offsets +
 *                   PA); primitives, triangles, materials and lights A's then B's, B's triangle, material and
 *                   `original` indices shifted by A's counts;
 *   G(lo, hi)       mesh lo when hi - lo == 1, else C(G(lo, mid), G(mid, hi)) with mid = lo + ceil((hi - lo) / 2): a
 *                   balanced tree over the meshes in slot order, each mesh the LBVH trace_scene_upload_mesh_device
 *                   builds (prims[k] = {TRIANGLE, order[k], tri_materials[order[k]], order[k]});
 *   D               C(base, G(0, k)): the meshes' triangles, materials and lights follow the base's in slot order, and
 *                   queries report triangle i of mesh j as Pb + n_0 + ... + n_{j-1} + i (Pb: the base's primitives)
 * - nodes, pair records, primitive and normal records, spheres, materials, lights, root reference, scene_scale and
 * counts alike.  A kept mesh enters D as the device holds it (with a refit's boxes and vertices).  The shadow tree is
 * composed, not rebuilt: C composes the parts' shadow trees the same way - pair 0 holds the two parts' root boxes and
 * references with C's split-axis bit, then A's pairs (pair references + 1), then B's (pair references + PA, leaf
 * references + PA): n_prims - 1 pairs, applied recursively through G.  The scene has one only when every part has one
 * (or is a single primitive), it has no spheres and the composed depth (1 + the deeper part's, per level) is at most
 * 64.  Answers do not depend on the shadow tree.
 * meshes[j] != NULL builds slot j from that descriptor (replacing or appending it); meshes[j] == NULL keeps the mesh
 * in slot j, which is not rebuilt: it costs a device copy with its references rebased when its place or its shifts
 * change, and nothing otherwise; nothing proportional to it crosses to the host.  Its shadow tree moves with it only
 * while option shadow_tree is on; a kept mesh moved with the option off has none until it is rebuilt (the scene then
 * has no shadow tree).  Slots from n_meshes on are dropped.  The call waits for the device a fixed number of times
 * whatever n_meshes is (the new meshes' build statuses are read back together).
 * The first attach after an upload moves the base's node, pair and shadow-pair records up one slot (a cost
 * proportional to the base, with a transient peak of about twice those buffers); later calls do not touch the base.
 * Memory: the build scratch holds every new mesh's LBVH build at once (each as trace_scene_upload_mesh_device's) and a
 * staging copy of the kept meshes that move; buffers only grow, so a repeated call with the same sizes allocates
 * nothing.  Refused before anything outside the build scratch is written (the previous scene and every slot stay as
 * they were, even when an earlier descriptor of the call was valid): the refusals of trace_scene_upload_mesh_device
 * for each new mesh, n_tris == 0, a new or kept mesh's tree deeper than 64 - ceil(log2 n_meshes) levels, n_meshes outside
 * [1, 64], a NULL descriptor for a slot that holds no mesh (every upload clears the slots), no scene uploaded, a base
 * without primitives, 2^30 or more primitives or too many interior nodes in the composed scene.
 * trace_scene_refit[_device] applies as after trace_scene_upload(D): its input is all triangles in D's order.  A
 * refit moves base and kept-mesh triangles until the next upload or replacement; a refit of a scene without a shadow
 * tree leaves the parts' shadow trees stale, so later calls compose none while such a part remains.  Like the uploads
 * the call drains all of the context's work, ends any SPPM session and is synchronous; it is local to the context
 * (every rank attaches the same meshes).  *n_nodes_out (may be NULL) receives the composed node count.
 * TRACE_BVH_PROFILE=1 prints per-phase times and the bytes staged for kept meshes. */
int trace_scene_attach_meshes_device(trace_ctx* ctx, int64_t n_meshes, const trace_mesh_device_desc* const* meshes,
                                     int64_t* n_nodes_out);
/* trace_scene_attach_meshes_device(ctx, 1, &mesh, n_nodes_out): the base with this one mesh. */
int trace_scene_attach_mesh_device(trace_ctx* ctx, const trace_mesh_device_desc* mesh, int64_t* n_nodes_out);

/* ---- refit (extension: the reference has no counterpart; it rebuilds BVHAccel).  New positions for the triangles of
 * the last upload, with the tree's topology kept (node structure, primitive order, materials, spheres, lights) and every
 * box recomputed on the GPU.  The result is exactly the scene trace_scene_upload would build from the same nodes and
 * primitives with the new vertices and these boxes:
 *   tri_vertices  [n_tris][3][3] world space, the triangle order of trace_scene_desc.tri_vertices; n_tris must be the
 *                 uploaded count.  The degenerate test is decided again (upload's unfused dot(g, g) == 0).
 *   tri_normals   same layout or NULL (keep the current normals); applied only to triangles uploaded with
 *                 TRACE_TRI_HAS_NORMALS.
 *   sphere_bounds [n_spheres][6] = min xyz, max xyz, host memory: the bounds the tree was built with (the spheres do not
 *                 move).  Required when the scene holds spheres, NULL otherwise.
 *   leaf box      Julia min / max (-0.0 < +0.0) union of its primitives' bounds (a triangle: its three vertices); a
 *                 zero-primitive leaf keeps its box and adds nothing to its parent's;
 *   interior box  Julia min / max union of its two children's boxes.  A refit with unchanged vertices therefore gives
 *                 back the uploaded boxes of the reference, sah and lbvh trees (float ==; the sign of a zero may differ);
 *   scene_scale   recomputed from the new root box with the upload's rule.
 * Refused, with the scene untouched: no scene uploaded, another triangle count, a scene with spheres and no (or the
 * wrong number of) sphere bounds, NaN in any vertex, normal or sphere bound.  The call first waits for all of the
 * context's work (an asynchronous SPPM session included) and ends any SPPM session, as trace_scene_upload does; it is
 * synchronous, so the caller may reuse its buffers on return.  Device buffers are rewritten in place: a captured Whitted
 * graph stays valid and replays over the new data (a changed scene_scale recaptures it).  Deterministic (bit-identical
 * for the same input); local to the context (no collectives: every rank refits with the same vertices).
 * TRACE_BVH_PROFILE=1 prints per-phase CUDA-event times to stderr. */
int trace_scene_refit(trace_ctx* ctx, int64_t n_tris, const float* tri_vertices, const float* tri_normals,
                      int64_t n_spheres, const float* sphere_bounds);
/* the same with vertices (and normals, or NULL) in device memory on the context's GPU, read on the context's stream:
 * the caller orders the work that wrote them before this call.  sphere_bounds stays in host memory. */
int trace_scene_refit_device(trace_ctx* ctx, int64_t n_tris, const void* tri_vertices_device,
                             const void* tri_normals_device, int64_t n_spheres, const float* sphere_bounds);
/* the uploaded scene's current nodes (n_nodes of the last upload), boxes as refit last left them */
int trace_scene_copy_nodes(trace_ctx* ctx, trace_bvh_node* nodes_out);
/* the uploaded scene's shadow tree: *n_pairs = its pair records (n_prims - 1), 0 when the scene has none (analytic
 * spheres, fewer than 2 primitives, a NaN vertex, deeper than 64 levels).  pairs_out (NULL: count only) receives
 * n_pairs x 64 bytes: per child {bmin.xyz, bmax.x} {bmax.y, bmax.z, reference, split-axis bit (first child) or 0};
 * reference = pair index, or 0x80000000 | primitive slot for a leaf.  Boxes as the last refit left them. */
int trace_scene_shadow_tree(trace_ctx* ctx, int64_t* n_pairs, void* pairs_out);
/* any-hit rays since the last trace_reset_stats that found a candidate occluder on the shadow tree which the exact
 * check could not confirm (or had a zero, tiny or non-finite direction component), and so were answered by the
 * reference tree's walk */
int trace_get_shadow_fallbacks(trace_ctx* ctx, uint64_t* out);
/* closest-hit rays since the last trace_reset_stats that the shadow-tree walk ("hit_tree") did not answer itself
 * (near tie of the two closest candidates, a check that failed, an irregular ray) and handed to the reference walk */
int trace_get_hit_fallbacks(trace_ctx* ctx, uint64_t* out);

/* ---- ray queries, host buffers. o,d: [n][3]; tmax_inout: [n] (t of the hit on return, unchanged on a miss);
 * prim_out: [n] original index + 1, 0 = miss; b0b1_out: [n][2] barycentrics (triangles) or 0; may be NULL. ---- */
int trace_intersect(trace_ctx* ctx, const float* o, const float* d, float* tmax_inout, int64_t n,
                    uint32_t* prim_out, float* b0b1_out);
int trace_occluded(trace_ctx* ctx, const float* o, const float* d, const float* tmax, int64_t n,
                   uint8_t* out);
/* device-resident variants: rays as two float4 arrays {o.xyz, t_max}, {d.xyz, unused}; hits float4 {t, prim+1 (bits), b0, b1} */
int trace_intersect_device(trace_ctx* ctx, const void* ray_o_tmax_device, const void* ray_d_device,
                           int64_t n, void* hit_out_device);
int trace_occluded_device(trace_ctx* ctx, const void* ray_o_tmax_device, const void* ray_d_device,
                          int64_t n, void* occluded_u8_out_device);

/* ---- Whitted (src/integrators/sampler.jl). film_xyzw: [crop_h][crop_w][4] = (X, Y, Z, filter_weight_sum),
 * accumulated into (the reference never clears the film, sampler.jl:52 / film.jl:182-193). ---- */
int trace_render_whitted(trace_ctx* ctx, const trace_camera* cam, const trace_film_desc* film,
                         int spp, int max_depth, uint64_t seed, float* film_xyzw_inout);
int trace_render_whitted_device(trace_ctx* ctx, const trace_camera* cam, const trace_film_desc* film,
                                int spp, int max_depth, uint64_t seed, void* film_xyzw_inout_device);

/* ---- SPPM (src/integrators/sppm.jl) ---- */
typedef void (*trace_sppm_cb)(void* user, int iteration, const float* rgb /* [crop_h][crop_w][3] */);
int trace_render_sppm(trace_ctx* ctx, const trace_camera* cam, const trace_film_desc* film,
                      float initial_radius, int max_depth, int n_iterations, int64_t photons_per_iteration,
                      int write_frequency, uint64_t seed, trace_sppm_cb on_image, void* user,
                      float* rgb_out /* [crop_h][crop_w][3], image after the last iteration (sppm.jl:461-472) */);
/* stepwise form used for multi-GPU sharding (options "rank"/"world" set BEFORE trace_sppm_begin): begin; per iteration
 * { [trace_photons(this rank's photon range): optional, asynchronous - the photon paths (sppm.jl:328-434 minus the
 *    deposits) then overlap the camera pass and the all-gather];
 *   camera_pass (this rank's image rows; with world == 1 it also builds the grid);
 *   [world > 1: all-gather buffers 2..6, then trace_sppm_build_grid];
 *   photon_pass(this rank's photon range); [world > 1: all-reduce(sum) buffer 0]; update };
 * [world > 1: all-gather buffer 1]; image; end.  Per-pixel buffers are in storage order: image rows dealt round-robin
 * to the ranks, each rank's rows contiguous (padded to ceil(H / world) rows), so rank r owns slice r of world. */
int   trace_sppm_begin(trace_ctx* ctx, const trace_camera* cam, const trace_film_desc* film,
                       float initial_radius, int max_depth, int64_t photons_per_iteration, uint64_t seed);
int   trace_sppm_camera_pass(trace_ctx* ctx, int iteration);
int   trace_sppm_trace_photons(trace_ctx* ctx, int iteration, int64_t photon_begin, int64_t photon_end);
int   trace_sppm_photon_pass(trace_ctx* ctx, int iteration, int64_t photon_begin, int64_t photon_end);
int   trace_sppm_build_grid(trace_ctx* ctx);
void* trace_sppm_flux_device(trace_ctx* ctx, int64_t* n_floats /* 4 per pixel slot: Phi.rgb, M */);
void* trace_sppm_buffer_device(trace_ctx* ctx, int which /* 0 flux, 1 Ld, 2..6 visible points */, int64_t* n_floats);
int   trace_sppm_update(trace_ctx* ctx);
int   trace_sppm_image(trace_ctx* ctx, int iteration, float* rgb_out);
int   trace_sppm_end(trace_ctx* ctx);
/* session form of trace_render_sppm's loop: after trace_sppm_begin, enqueue iterations first .. first + n - 1 back to
 * back (no host wait; with a communicator the all-gather / all-reduce of every iteration run inside); read the image
 * with trace_sppm_image (which waits and reports any queue / grid overflow), finish with trace_sppm_end. */
int   trace_sppm_iterate(trace_ctx* ctx, int first_iteration, int n);

#ifdef __cplusplus
}
#endif
#endif /* TRACE_CUDA_H */
