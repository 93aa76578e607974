// sppm.cu — Stochastic Progressive Photon Mapping on the same wavefront stages as whitted.cu.
//
// Replaces src/integrators/sppm.jl:132-569: _generate_visible_sppm_points! (camera pass), _clean_grid! +
// _populate_grid! (hash grid of visible points), _trace_photons! (photon pass with deposits), _update_pixels! and
// _sppm_to_image.  Quirks kept (SURVEY.md §9): Q7 photon beta never updated, Q8 Ld not multiplied by beta, Q9 tau
// update without vp.beta and N / radius in Float64, Q10 a visible point sits in every hashed cell its +-r box
// overlaps (duplicates kept) and the hash is evaluated in UInt64, Q22 default photon count, Q23 visible-point rule.
//
// Data layout: per-pixel state as float4 arrays; the reference's per-cell linked lists become a CSR table
// (cell_start[n_pixels+1], cell_items[]) rebuilt each iteration by count -> scan -> fill; deposits are one 128-bit
// vector atomic (Phi.rgb, M) per accepted visible point.  The flux buffer is what multi-GPU runs all-reduce.
#include "context.hpp"
#include "shading.cuh"
#include "wavefront.cuh"

struct GridParams {
    float lo[3], hi[3];
    float max_radius;
    int res[3];
    int valid;
    unsigned int total_items;
};

struct SppmLaunch {
    DeviceScene sc;
    DeviceCamera cam;
    DeviceFilm film;
    int max_depth, iteration;
    uint64_t seed;
    int W, H, npix;            // npix = W*H is also the hash-table size (sppm.jl:141)
    unsigned long long hash_magic;   // h % npix without a 64-bit division: q = mulhi(h, magic) >> shift (grid_hash)
    int hash_shift;                  // < 0: tables of <= 64 cells take the plain modulo
    // pixel STORAGE order (all per-pixel arrays): image rows are dealt round-robin to `world` ranks and each rank's rows
    // are contiguous, padded to chunk_rows rows - so a rank's visible points are one slice that an all-gather can move.
    // world == 1: storage index == raster index.
    int world, rank, chunk_rows, nstore;
    long long photons_per_iteration;
    // per-pixel state
    float4* Ld;        // rgb
    float4* flux;      // Phi.rgb, M
    float4* tau_r;     // tau.rgb, radius
    double* N;
    float4 *vpA, *vpB, *vpC, *vpD, *vpE;   // {p, r^2} {wo, material} {ns, valid} {ss, -} {ng, -}
    // grid
    GridParams* grid;
    unsigned int *cell_start, *cell_cursor, *cell_items;
    float4* cell_vp;           // {p, r^2} of each CSR entry, in list order: candidate tests stream 16 B coalesced
    unsigned int items_cap;
    // queues
    float4 *ro[2], *rd[2], *rw[2], *hits;
    float4 *so, *sd, *sc_contrib;
    int* counters;             // this lane's queue counters
    int* flags;                // [IC_OVERFLOW], [IC_ERROR]: one pair for the whole session (lane 0's block)
    int cap;
    int cap_shadow;            // shadow-ray queue (camera pass) / deposit-request queue (photon pass): all levels share it
    int range_begin, range_end;   // camera pass: the storage slots this lane generates paths for
    // photons
    long long photon_begin;    // first photon index (within the iteration) of this launch
    int n_photons;
    const float* light_cdf;    // n_lights + 1
    const float* light_func;   // n_lights
    float light_func_int;
    unsigned long long* stats;
};

__device__ __forceinline__ bool storage_to_raster(const SppmLaunch& L, int s, int& x, int& y) {
    const int row = s / L.W;
    x = s - row * L.W;
    const int owner = row / L.chunk_rows, local = row - owner * L.chunk_rows;
    y = local * L.world + owner;
    return y < L.H;                       // false: padding slot
}
__device__ __forceinline__ int raster_to_storage(const SppmLaunch& L, int x, int y) {
    return ((y % L.world) * L.chunk_rows + y / L.world) * L.W + x;
}

// ---------------------------------------------------------------- camera pass
// One camera path per pixel of THIS rank's rows (sppm.jl:184-196). The RNG is keyed by the raster pixel index, so the
// visible points do not depend on the number of ranks.
// the camera ray of storage slot `st` (false: padding slot); the RNG is keyed by the raster pixel
__device__ __forceinline__ bool cam_generate_ray(const SppmLaunch& L, int st, int& pix, float3& o, float3& d) {
    int x, y;
    if (!storage_to_raster(L, st, x, y)) return false;
    pix = y * L.W + x;      // raster index: RNG key
    const int px = L.film.crop_x0 + x, py = L.film.crop_y0 + y;
    const uint32_t it = (uint32_t)L.iteration;
    const float u0 = rng_uniform(L.seed, (uint32_t)pix, it, 0), u1 = rng_uniform(L.seed, (uint32_t)pix, it, 1);
    float l0 = 0.0f, l1 = 0.0f;
    if (L.cam.lens_radius > 0.0f) { l0 = rng_uniform(L.seed, (uint32_t)pix, it, 2); l1 = rng_uniform(L.seed, (uint32_t)pix, it, 3); }
    generate_camera_ray(L.cam, (float)px + u0, (float)py + u1, l0, l1, o, d);
    return true;
}

__global__ void __launch_bounds__(256) k_sppm_cam_generate(SppmLaunch L) {
    for (int st = L.range_begin + blockIdx.x * blockDim.x + threadIdx.x; st < L.range_end; st += gridDim.x * blockDim.x) {
        int pix = 0;
        float3 o = f3s(0.0f), d = f3s(1.0f);
        // no compaction at level 1: queue slot = path index (one same-address atomic per warp costs more than the few
        // padding slots, which get a ray that cannot hit anything: t_max < 0)
        const bool live = cam_generate_ray(L, st, pix, o, d);
        const int q = st - L.range_begin;
        if (st == L.range_end - 1) L.counters[1] = L.range_end - L.range_begin;
        L.ro[0][q] = f4(o, live ? TR_INF : -1.0f);
        L.rd[0][q] = f4(d, __int_as_float(st));          // the path carries its STORAGE slot
        L.rw[0][q] = make_float4(1.0f, 1.0f, 1.0f, __int_as_float(pix));   // ... and its raster index (RNG key)
    }
}

// One camera-path vertex (sppm.jl:204-266): direct lighting (a shadow ray into the pass's shadow queue), visible point
// or continuation.  Returns true when the path continues with (o, d, beta) updated.  Shared by the wavefront kernel
// (one launch per bounce level) and the path kernel (all levels in one launch), so both compute the same bits.
__device__ __forceinline__ bool cam_shade_ray(const SppmLaunch& L, int level, float4 h, float3& o, float3& d, float3& beta, int slot, int pix) {
    if (d.x == 0.0f) d.x = 0.0f;
    if (d.y == 0.0f) d.y = 0.0f;
    if (d.z == 0.0f) d.z = 0.0f;
    const uint32_t prim = __float_as_uint(h.y) - 1u;
    const float b2 = third_barycentric(L.sc, prim, o, d);
    const Interaction it = build_interaction(L.sc, prim, o, d, h.z, h.w, b2);
    const Frame fr = make_frame(it);
    LobeSet lobes;
    material_lobes(L.sc.materials[it.material], true, lobes);
    const float3 wo = -d;
    const uint32_t dim = 5u + 8u * (uint32_t)(level - 1), itn = (uint32_t)L.iteration;
    // uniform_sample_one_light + estimate_direct (sppm.jl:503-554); NOT multiplied by beta (Q8)
    {
        const int nl = L.sc.n_lights;
        const float ul = rng_uniform(L.seed, (uint32_t)pix, itn, dim + 0);
        const int ln = max(1, min((int)ceilf(ul * (float)nl), nl));
        const float light_pdf = 1.0f / (float)nl;
        float3 wi, lpos;
        const float3 Li = sample_li_any(L.sc.lights[ln - 1], it.p, wi, lpos);
        if (!is_black3(Li)) {
            const float3 f = bsdf_f(lobes, fr, it.wo, wi, LB_ALL & ~LB_SPECULAR) * fabsf(dot3(wi, it.ns));
            if (!is_black3(f)) {
                const float3 contrib = ((f * Li) / 1.0f) / light_pdf;
                const float3 sdir = lpos - it.p;
                const int q = queue_claim(&L.counters[32]);
                if (q >= L.cap_shadow) { L.flags[IC_OVERFLOW_SHADOW] = 1; return false; }
                L.so[q] = f4(it.p + 1e-6f * sdir, TR_INF);
                L.sd[q] = f4(sdir, __int_as_float(slot));
                L.sc_contrib[q] = f4(contrib, 0.0f);
            }
        }
    }
    const bool is_diffuse = num_components(lobes, LB_DIFFUSE | LB_REFLECTION | LB_TRANSMISSION) > 0;
    const bool is_glossy = num_components(lobes, LB_GLOSSY | LB_REFLECTION | LB_TRANSMISSION) > 0;
    if (is_diffuse || (is_glossy && level == L.max_depth)) {
        // (the search radius is attached when the grid is built: the camera pass must not depend on the previous
        // iteration's update, so that it can run ahead of it - see the pipeline in sppm_iteration_async)
        L.vpA[slot] = f4(it.p, 0.0f);
        L.vpB[slot] = f4(wo, __uint_as_float(it.material));
        L.vpC[slot] = f4(fr.ns, is_black3(beta) ? 0.0f : 1.0f);
        L.vpD[slot] = f4(fr.ss, 0.0f);
        L.vpE[slot] = f4(fr.ng, 0.0f);
        return false;
    }
    if (level == L.max_depth) return false;
    const BSDFSample bs = bsdf_sample(lobes, fr, wo, rng_uniform(L.seed, (uint32_t)pix, itn, dim + 5),
                                      rng_uniform(L.seed, (uint32_t)pix, itn, dim + 6), LB_ALL);
    if (bs.pdf == 0.0f || is_black3(bs.f)) return false;
    beta = beta * (bs.f * fabsf(dot3(bs.wi, it.ns)) / bs.pdf);
    const float by = luminance(beta);
    if (by < 0.25f) {
        const float cp = fminf(1.0f, by);
        if (rng_uniform(L.seed, (uint32_t)pix, itn, dim + 7) > cp) return false;
        beta = beta / cp;
    }
    o = it.p + 1e-6f * bs.wi;
    d = bs.wi;
    return true;
}

#ifndef TR_SPPM_SHADE_MIN_BLOCKS
#define TR_SPPM_SHADE_MIN_BLOCKS 8
#endif
__global__ void __launch_bounds__(128, TR_SPPM_SHADE_MIN_BLOCKS) k_sppm_cam_shade(SppmLaunch L, int level) {
    const int cur = (level - 1) & 1, nxt = level & 1;
    const int n = min(L.counters[level], L.cap);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 h = L.hits[i];
        if (__float_as_uint(h.y) == 0u) continue;
        const float4 o4 = L.ro[cur][i], d4 = L.rd[cur][i], w4 = L.rw[cur][i];
        float3 o = xyz(o4), d = xyz(d4), beta = xyz(w4);
        const int slot = __float_as_int(d4.w);      // storage slot of the pixel
        const int pix = __float_as_int(w4.w);       // raster index: RNG key
        if (!cam_shade_ray(L, level, h, o, d, beta, slot, pix)) continue;
        const int q = queue_claim(&L.counters[level + 1]);
        L.ro[nxt][q] = f4(o, TR_INF);
        L.rd[nxt][q] = f4(d, __int_as_float(slot));
        L.rw[nxt][q] = f4(beta, __int_as_float(pix));
    }
}

// Path kernel: one thread carries one camera path through its first `path_levels` bounces - generate, then (closest hit
// -> vertex) - without ray queues in HBM; the paths that are still alive afterwards enter the wavefront queues of the next
// level.  Measured (profiles/r2_experiments.md): carrying paths through ALL levels in one kernel is 1.7-3x SLOWER than the
// wavefront (only the few lanes whose path hit glass stay alive at deeper levels, un-compacted: 3-10 of 32 lanes walk
// the 600-node glass block), so the default is path_levels = 1: the level where every lane has a ray - generate, extend
// and shade of the largest level in one launch, no primary-ray / hit queues - and compacted queues from level 2 on.
// Every vertex goes through cam_shade_ray, so visible points and shadow rays are those of the wavefront kernels.
#ifndef TR_PATH_MIN_BLOCKS
#define TR_PATH_MIN_BLOCKS 6
#endif
static __device__ __noinline__ bool cam_vertex(const SppmLaunch& L, int level, float4 h, float3& o, float3& d, float3& beta, int slot, int pix) {
    return cam_shade_ray(L, level, h, o, d, beta, slot, pix);
}
static __device__ __noinline__ bool cam_first_ray(const SppmLaunch& L, int st, int& pix, float3& o, float3& d) {
    return cam_generate_ray(L, st, pix, o, d);
}
template <int SLAB, bool COUNT, int WAIT, bool TREE>       // TREE: walk the shadow tree (traverse_closest)
__global__ void __launch_bounds__(128, TR_PATH_MIN_BLOCKS) k_sppm_cam_path(const __grid_constant__ SppmLaunch L, int path_levels, int* error_flag) {
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    unsigned n_rays = 0;
    for (int base = L.range_begin + blockIdx.x * blockDim.x + (threadIdx.x - lane); base < L.range_end; base += gridDim.x * blockDim.x) {
        const int st = base + lane;
        int pix = 0;
        float3 o = f3s(0.0f), d = f3s(1.0f), beta = f3s(1.0f);
        bool alive = st < L.range_end && cam_first_ray(L, st, pix, o, d);
        const int last = min(L.max_depth, path_levels);
        for (int level = 1; level <= last; ++level) {
            __syncwarp();                                         // reconverge before the walk (see k_wh_primary)
            if (!__any_sync(full, alive)) break;
            HitRecord h;
            traverse_closest<SLAB, COUNT, WAIT, TREE>(L.sc, alive, o, d, TR_INF, h, L.stats + ST_NODES, error_flag);
            if (alive) {
                n_rays++;
                alive = h.prim != 0u && cam_vertex(L, level, make_float4(h.t, __uint_as_float(h.prim), h.b0, h.b1), o, d, beta, st, pix);
            }
        }
        if (alive && last < L.max_depth) {                        // the rest of the path goes through the wavefront queues
            const int q = queue_claim(&L.counters[last + 1]);
            L.ro[last & 1][q] = f4(o, TR_INF);
            L.rd[last & 1][q] = f4(d, __int_as_float(st));
            L.rw[last & 1][q] = f4(beta, __int_as_float(pix));
        }
    }
    __syncwarp();
    n_rays = __reduce_add_sync(full, n_rays);
    if (lane == 0 && n_rays) atomicAdd(&L.stats[ST_RAYS_EXTEND], (unsigned long long)n_rays);
}

// ---------------------------------------------------------------- grid build (sppm.jl:278-318)
__device__ __forceinline__ void atomic_min_float(float* a, float v) {
    if (v >= 0.0f) atomicMin((int*)a, __float_as_int(v)); else atomicMax((unsigned int*)a, __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_float(float* a, float v) {
    if (v >= 0.0f) atomicMax((int*)a, __float_as_int(v)); else atomicMin((unsigned int*)a, __float_as_uint(v));
}

__global__ void k_grid_reset(GridParams* g) {
    for (int k = 0; k < 3; ++k) { g->lo[k] = TR_INF; g->hi[k] = -TR_INF; g->res[k] = 1; }
    g->max_radius = 0.0f; g->valid = 0; g->total_items = 0;
}

__global__ void __launch_bounds__(256) k_grid_bounds(SppmLaunch L) {
    float lo[3] = {TR_INF, TR_INF, TR_INF}, hi[3] = {-TR_INF, -TR_INF, -TR_INF}, mr = 0.0f;
    for (int pix = blockIdx.x * blockDim.x + threadIdx.x; pix < L.nstore; pix += gridDim.x * blockDim.x) {
        if (L.vpC[pix].w == 0.0f) continue;                       // is_black(vp.beta)
        const float4 A = L.vpA[pix];
        const float r = L.tau_r[pix].w;
        lo[0] = fminf(lo[0], A.x - r); lo[1] = fminf(lo[1], A.y - r); lo[2] = fminf(lo[2], A.z - r);   // expand(Bounds3(p), r)
        hi[0] = fmaxf(hi[0], A.x + r); hi[1] = fmaxf(hi[1], A.y + r); hi[2] = fmaxf(hi[2], A.z + r);
        mr = fmaxf(mr, r);
    }
    for (int off = 16; off > 0; off >>= 1) {
        for (int k = 0; k < 3; ++k) {
            lo[k] = fminf(lo[k], __shfl_xor_sync(0xffffffffu, lo[k], off));
            hi[k] = fmaxf(hi[k], __shfl_xor_sync(0xffffffffu, hi[k], off));
        }
        mr = fmaxf(mr, __shfl_xor_sync(0xffffffffu, mr, off));
    }
    // one set of atomics per CTA, not per warp: all of them hit the same seven words (ncu: 48 us at 8 % issue utilisation
    // for a 40 MB read - serialised same-address atomics)
    __shared__ float s_red[8][7];
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { for (int k = 0; k < 3; ++k) { s_red[w][k] = lo[k]; s_red[w][3 + k] = hi[k]; } s_red[w][6] = mr; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int j = 1; j < (int)(blockDim.x >> 5); ++j) {
            for (int k = 0; k < 3; ++k) { lo[k] = fminf(lo[k], s_red[j][k]); hi[k] = fmaxf(hi[k], s_red[j][3 + k]); }
            mr = fmaxf(mr, s_red[j][6]);
        }
        if (mr > 0.0f) {
            for (int k = 0; k < 3; ++k) { atomic_min_float(&L.grid->lo[k], lo[k]); atomic_max_float(&L.grid->hi[k], hi[k]); }
            atomic_max_float(&L.grid->max_radius, mr);
        }
    }
}

__global__ void k_grid_params(GridParams* g) {                    // sppm.jl:293-301
    if (!(g->max_radius > 0.0f)) { g->valid = 0; return; }
    const float dx = g->hi[0] - g->lo[0], dy = g->hi[1] - g->lo[1], dz = g->hi[2] - g->lo[2];
    const float max_diag = fmaxf(fmaxf(dx, dy), dz);
    const long long base = (long long)floorf(max_diag / g->max_radius);
    const float dg[3] = {dx, dy, dz};
    for (int k = 0; k < 3; ++k) {
        long long r = (long long)floorf((float)base * dg[k] / max_diag);
        g->res[k] = (int)max(1ll, min(r, 1ll << 30));
    }
    g->valid = 1;
}

// to_grid (sppm.jl:479-495): returns in_bounds, writes the clamped cell
__device__ __forceinline__ bool to_grid(const GridParams& g, float3 p, int cell[3]) {
    const float o[3] = {p.x - g.lo[0], p.y - g.lo[1], p.z - g.lo[2]};          // offset(bounds, p), bounds.jl:134-143
    const bool gx = g.hi[0] > g.lo[0], gy = g.hi[1] > g.lo[1], gz = g.hi[2] > g.lo[2];
    const bool gg[3] = {gx, gy, gz};
    bool in = true;
    for (int k = 0; k < 3; ++k) {
        float off = o[k];
        if (gx || gy || gz) off = off / (gg[k] ? g.hi[k] - g.lo[k] : 1.0f);
        const float f = floorf((float)g.res[k] * off);
        // Int64(floor(...)) then 0 <= c < res
        if (!(f >= 0.0f && f < (float)g.res[k])) in = false;
        const float cl = fminf(fmaxf(f, 0.0f), (float)(g.res[k] - 1));
        cell[k] = (f != f) ? 0 : (int)cl;
    }
    return in;
}
// sppm.jl:497-501, UInt64 math (Q10).  Cell coordinates are < 2^30, so h < 2^57; with L = ceil(log2 size), k = 57 + L and
// magic = ceil(2^k / size) (< 2^58 + 1), floor(h * magic / 2^k) == floor(h / size) exactly (error h * e / 2^k < 1 / size for
// e < 1) - one 64x64 high multiply instead of the ~100-instruction 64-bit modulo that dominated k_grid_insert.
__device__ __forceinline__ unsigned int grid_hash(int x, int y, int z, const SppmLaunch& L) {
    const unsigned long long h = ((unsigned long long)x * 73856093ull) ^ ((unsigned long long)y * 19349663ull) ^
                                 ((unsigned long long)z * 83492791ull);
    if (L.hash_shift < 0) return (unsigned int)(h % (unsigned long long)(unsigned int)L.npix);
    const unsigned long long q = __umul64hi(h, L.hash_magic) >> L.hash_shift;
    return (unsigned int)(h - q * (unsigned long long)(unsigned int)L.npix);
}

template <bool FILL>
__global__ void __launch_bounds__(256) k_grid_insert(SppmLaunch L) {
    const GridParams g = *L.grid;
    if (!g.valid) return;
    const int lane = threadIdx.x & 31;
    for (int pix = blockIdx.x * blockDim.x + threadIdx.x; pix < L.nstore; pix += gridDim.x * blockDim.x) {
        if (L.vpC[pix].w == 0.0f) continue;
        const float4 A = L.vpA[pix];
        const float r = L.tau_r[pix].w;
        int c0[3], c1[3];
        to_grid(g, f3(A.x - r, A.y - r, A.z - r), c0);
        to_grid(g, f3(A.x + r, A.y + r, A.z + r), c1);
        for (int z = c0[2]; z <= c1[2]; ++z) for (int y = c0[1]; y <= c1[1]; ++y) for (int x = c0[0]; x <= c1[0]; ++x) {
            const unsigned int h = grid_hash(x, y, z, L);
            // neighbouring pixels fall into the same cells (a cell holds thousands of visible points where the pixel
            // footprint is far below the radius): the lanes that hit the same cell right now issue ONE atomic
            const unsigned int active = __activemask();
            const unsigned int peers = __match_any_sync(active, h);
            const int leader = __ffs(peers) - 1;
            const unsigned int n_peers = (unsigned int)__popc(peers);
            if (!FILL) { if (lane == leader) atomicAdd(&L.cell_start[h], n_peers); }
            else {
                unsigned int base = 0;
                if (lane == leader) base = atomicAdd(&L.cell_cursor[h], n_peers);
                base = __shfl_sync(peers, base, leader);
                const unsigned int slot = base + (unsigned int)__popc(peers & ((1u << lane) - 1u));
                if (slot < L.items_cap) { L.cell_items[slot] = (unsigned int)pix; L.cell_vp[slot] = make_float4(A.x, A.y, A.z, r * r); }
            }
        }
    }
}

// exclusive scan of cell_start[0..n) in three small kernels (block scan, scan of block sums, add)
#define SCAN_BLOCK 1024
#define SCAN_ITEMS 4
__global__ void __launch_bounds__(SCAN_BLOCK) k_scan_blocks(unsigned int* data, int n, unsigned int* block_sums) {
    __shared__ unsigned int warp_sums[32];
    const int base = blockIdx.x * SCAN_BLOCK * SCAN_ITEMS + threadIdx.x * SCAN_ITEMS;
    unsigned int v[SCAN_ITEMS], sum = 0;
    for (int k = 0; k < SCAN_ITEMS; ++k) { v[k] = (base + k < n) ? data[base + k] : 0u; sum += v[k]; }
    unsigned int incl = sum;
    for (int off = 1; off < 32; off <<= 1) { unsigned int t = __shfl_up_sync(0xffffffffu, incl, off); if ((threadIdx.x & 31) >= off) incl += t; }
    if ((threadIdx.x & 31) == 31) warp_sums[threadIdx.x >> 5] = incl;
    __syncthreads();
    if (threadIdx.x < 32) {
        unsigned int w = warp_sums[threadIdx.x], wi = w;
        for (int off = 1; off < 32; off <<= 1) { unsigned int t = __shfl_up_sync(0xffffffffu, wi, off); if (threadIdx.x >= off) wi += t; }
        warp_sums[threadIdx.x] = wi - w;
        if (threadIdx.x == 31) block_sums[blockIdx.x] = wi;
    }
    __syncthreads();
    unsigned int excl = warp_sums[threadIdx.x >> 5] + incl - sum;
    for (int k = 0; k < SCAN_ITEMS; ++k) { if (base + k < n) data[base + k] = excl; excl += v[k]; }
}
__global__ void k_scan_sums(unsigned int* block_sums, int n_blocks, GridParams* g) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        unsigned int acc = 0;
        for (int i = 0; i < n_blocks; ++i) { unsigned int t = block_sums[i]; block_sums[i] = acc; acc += t; }
        g->total_items = acc;
    }
}
__global__ void __launch_bounds__(SCAN_BLOCK) k_scan_add(unsigned int* data, int n, const unsigned int* block_sums, unsigned int* cursor) {
    const int base = blockIdx.x * SCAN_BLOCK * SCAN_ITEMS + threadIdx.x * SCAN_ITEMS;
    const unsigned int add = block_sums[blockIdx.x];
    for (int k = 0; k < SCAN_ITEMS; ++k) if (base + k < n) { unsigned int v = data[base + k] + add; data[base + k] = v; cursor[base + k] = v; }
}
__global__ void k_grid_check(SppmLaunch L) {
    if (L.grid->total_items > L.items_cap) L.flags[IC_OVERFLOW] = 1;
    L.cell_start[L.npix] = L.grid->total_items;
    atomicAdd(&L.stats[ST_GRID_ITEMS], (unsigned long long)L.grid->total_items);
}

// ---------------------------------------------------------------- photon pass (sppm.jl:320-436)
// photon j of this launch: light choice, direction and initial beta (sppm.jl:334-360).  False: the photon carries nothing.
__device__ __forceinline__ bool photon_generate_ray(const SppmLaunch& L, int j, float3& o, float3& d, float3& beta) {
    const unsigned long long hidx = (unsigned long long)(L.iteration - 1) * (unsigned long long)L.photons_per_iteration +
                                    (unsigned long long)(L.photon_begin + j);
    // light choice: sample_discrete(light_distribution, halton dim 0), sampling.jl:32-41
    const float ls = radical_inverse(0, hidx);
    const int nl = L.sc.n_lights;
    int last = -1;
    for (int k = 0; k <= nl; ++k) if (L.light_cdf[k] <= ls) last = k;
    const int ln = min(max(last, 0), nl - 1);
    const float light_pdf = L.light_func_int > 0.0f ? L.light_func[ln] / (L.light_func_int * (float)nl) : 0.0f;
    const DeviceLight& light = L.sc.lights[ln];
    const float u0 = radical_inverse(1, hidx), u1 = radical_inverse(2, hidx);
    // sample_le (point.jl:60-69, spot.jl:46-55)
    float3 le;
    float pdf_dir;
    const float3 I = f3(light.I[0], light.I[1], light.I[2]);
    if (light.kind == TRACE_LIGHT_POINT) { d = uniform_sphere(u0, u1); pdf_dir = 1.0f / (4.0f * TR_PI); le = I; }
    else {
        d = xform_vector(light.m, uniform_cone(u0, u1, light.cos_total));
        pdf_dir = 1.0f / (2.0f * TR_PI * (1.0f - light.cos_total));
        le = I * spot_falloff(light, d);
    }
    const float pdf_pos = 1.0f;
    if (pdf_dir == 0.0f || is_black3(le)) return false;
    beta = (fabsf(dot3(d, d)) * le) / (light_pdf * pdf_pos * pdf_dir);      // light_normal == ray.d
    if (is_black3(beta)) return false;
    o = f3(light.pos[0], light.pos[1], light.pos[2]);
    return true;
}

__global__ void __launch_bounds__(256) k_photon_generate(SppmLaunch L) {
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < L.n_photons; j += gridDim.x * blockDim.x) {
        float3 o = f3s(0.0f), d = f3s(1.0f), beta = f3s(0.0f);
        const bool live = photon_generate_ray(L, j, o, d, beta);
        const int q = j;                                  // (see k_sppm_cam_generate)
        if (j == L.n_photons - 1) L.counters[1] = L.n_photons;
        L.ro[0][q] = f4(o, live ? TR_INF : -1.0f);
        L.rd[0][q] = f4(d, __int_as_float(j));
        L.rw[0][q] = f4(beta, luminance(beta));
    }
}

// One photon-path vertex (sppm.jl:362-434): a deposit request at depth > 1, then the continuation.  beta is NOT updated
// along the path (Q7); `lum0` = Y(beta).  Returns true when the photon flies on with (o, d) updated.
__device__ __forceinline__ bool photon_shade_ray(const SppmLaunch& L, int level, float4 h, float3& o, float3& d, float3 beta, float lum0, int j) {
    if (d.x == 0.0f) d.x = 0.0f;
    if (d.y == 0.0f) d.y = 0.0f;
    if (d.z == 0.0f) d.z = 0.0f;
    const uint32_t prim = __float_as_uint(h.y) - 1u;
    const float b2 = third_barycentric(L.sc, prim, o, d);
    const Interaction it = build_interaction(L.sc, prim, o, d, h.z, h.w, b2);
    const float3 wo = -d;
    if (level > 1) {
        // photon landed at depth > 1: queue a deposit request for k_photon_deposit (sppm.jl:377-403).  The grid is
        // NOT consulted here - it is being rebuilt by the concurrent camera pass; the deposit kernel does the lookup
        const int q = queue_claim(&L.counters[32]);
        if (q >= L.cap_shadow) { L.flags[IC_OVERFLOW_DEPOSIT] = 1; return false; }
        L.so[q] = f4(it.p, 0.0f);
        L.sd[q] = f4(wo, 0.0f);
        L.sc_contrib[q] = f4(beta, 0.0f);
    }
    const Frame fr = make_frame(it);
    LobeSet lobes;
    material_lobes(L.sc.materials[it.material], true, lobes);
    const unsigned long long hidx = (unsigned long long)(L.iteration - 1) * (unsigned long long)L.photons_per_iteration +
                                    (unsigned long long)(L.photon_begin + j);
    const int hdim = 6 + 3 * (level - 1);
    const BSDFSample bs = bsdf_sample(lobes, fr, wo, radical_inverse(hdim, hidx), radical_inverse(hdim + 1, hidx), LB_ALL);
    if (is_black3(bs.f) || bs.pdf == 0.0f) return false;
    const float3 beta_new = ((beta * bs.f) * fabsf(dot3(bs.wi, it.ns))) / bs.pdf;
    const float q = fmaxf(0.0f, 1.0f - luminance(beta_new) / lum0);
    if (radical_inverse(hdim + 2, hidx) < q) return false;
    if (level + 1 > L.max_depth) return false;
    o = it.p + 1e-6f * bs.wi;
    d = bs.wi;
    return true;
}

__global__ void __launch_bounds__(128, TR_SPPM_SHADE_MIN_BLOCKS) k_photon_shade(SppmLaunch L, int level) {
    const int cur = (level - 1) & 1, nxt = level & 1;
    const int n = min(L.counters[level], L.cap);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 h = L.hits[i];
        if (__float_as_uint(h.y) == 0u) continue;
        const float4 o4 = L.ro[cur][i], d4 = L.rd[cur][i], w4 = L.rw[cur][i];
        float3 o = xyz(o4), d = xyz(d4);
        if (!photon_shade_ray(L, level, h, o, d, xyz(w4), w4.w, __float_as_int(d4.w))) continue;
        const int qi = queue_claim(&L.counters[level + 1]);
        L.ro[nxt][qi] = f4(o, TR_INF);
        L.rd[nxt][qi] = f4(d, d4.w);
        L.rw[nxt][qi] = w4;                                      // beta is NOT updated (Q7)
    }
}

// photon path kernel: see k_sppm_cam_path
static __device__ __noinline__ bool photon_vertex(const SppmLaunch& L, int level, float4 h, float3& o, float3& d, float3 beta, float lum0, int j) {
    return photon_shade_ray(L, level, h, o, d, beta, lum0, j);
}
static __device__ __noinline__ bool photon_first_ray(const SppmLaunch& L, int j, float3& o, float3& d, float3& beta) {
    return photon_generate_ray(L, j, o, d, beta);
}
template <int SLAB, bool COUNT, int WAIT, bool TREE>       // TREE: walk the shadow tree (traverse_closest)
__global__ void __launch_bounds__(128, TR_PATH_MIN_BLOCKS) k_photon_path(const __grid_constant__ SppmLaunch L, int path_levels, int* error_flag) {
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    unsigned n_rays = 0;
    for (int base = blockIdx.x * blockDim.x + (threadIdx.x - lane); base < L.n_photons; base += gridDim.x * blockDim.x) {
        const int j = base + lane;
        float3 o = f3s(0.0f), d = f3s(1.0f), beta = f3s(0.0f);
        bool alive = j < L.n_photons && photon_first_ray(L, j, o, d, beta);
        const float lum0 = luminance(beta);
        const int last = min(L.max_depth, path_levels);
        for (int level = 1; level <= last; ++level) {
            __syncwarp();
            if (!__any_sync(full, alive)) break;
            HitRecord h;
            traverse_closest<SLAB, COUNT, WAIT, TREE>(L.sc, alive, o, d, TR_INF, h, L.stats + ST_NODES, error_flag);
            if (alive) {
                n_rays++;
                alive = h.prim != 0u && photon_vertex(L, level, make_float4(h.t, __uint_as_float(h.prim), h.b0, h.b1), o, d, beta, lum0, j);
            }
        }
        if (alive && last < L.max_depth) {
            const int q = queue_claim(&L.counters[last + 1]);
            L.ro[last & 1][q] = f4(o, TR_INF);
            L.rd[last & 1][q] = f4(d, __int_as_float(j));
            L.rw[last & 1][q] = f4(beta, lum0);
        }
    }
    __syncwarp();
    n_rays = __reduce_add_sync(full, n_rays);
    if (lane == 0 && n_rays) atomicAdd(&L.stats[ST_RAYS_EXTEND], (unsigned long long)n_rays);
}

// One WARP per deposit request: the 32 lanes stride over the hashed cell's CSR list (coalesced index loads), test
// |vp.p - p|^2 <= r^2 and, for accepted visible points, evaluate vp.bsdf(vp.wo, -d) and add (beta * f, 1) to
// (Phi, M) with one 128-bit vector atomic.  Lists are long where visible points are dense (cell edge ~ max radius,
// pixel footprint << radius: thousands of entries per cell), so a thread-per-photon loop serialises on its longest
// list; a warp per request keeps every lane busy and the loads coalesced.
#define TR_DEPOSIT_SPLIT 8
__global__ void __launch_bounds__(128) k_photon_deposit(SppmLaunch L, int level) {
    const int n = min(L.counters[32], L.cap_shadow);
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    unsigned int deposits = 0, candidates = 0;
    // TR_DEPOSIT_SPLIT warps share one request (interleaved 32-entry slices of its list): a request's chain of
    // dependent gathers is 8x shorter and there are 8x more independent tasks to hide latency with
    const long long n_tasks = (long long)n * TR_DEPOSIT_SPLIT;
    const GridParams g = *L.grid;
    if (!g.valid) return;
    for (long long task = warp; task < n_tasks; task += n_warps) {
        const int r = (int)(task / TR_DEPOSIT_SPLIT), sub = (int)(task % TR_DEPOSIT_SPLIT);
        const float3 p = xyz(L.so[r]);
        int cell[3];
        if (!to_grid(g, p, cell)) continue;
        const unsigned int hsh = grid_hash(cell[0], cell[1], cell[2], L);
        const unsigned int e0 = L.cell_start[hsh], e1 = L.cell_start[hsh + 1];
        if (e0 + sub * 32 >= e1) continue;
        const float3 wo = xyz(L.sd[r]), beta = xyz(L.sc_contrib[r]);
        for (unsigned int e = e0 + sub * 32 + lane; e < e1; e += 32 * TR_DEPOSIT_SPLIT) {
            const float4 A = __ldcs(&L.cell_vp[e]);                  // streamed once per request: keep it out of L1
            candidates++;
            const float3 dd = xyz(A) - p;
            if (dot3(dd, dd) > A.w) continue;
            const unsigned int pix = L.cell_items[e];
            const float4 Bv = L.vpB[pix];
            Frame vf;
            vf.ns = xyz(L.vpC[pix]); vf.ss = xyz(L.vpD[pix]); vf.ng = xyz(L.vpE[pix]);
            vf.ts = cross3(vf.ns, vf.ss);
            LobeSet vl;
            material_lobes(L.sc.materials[__float_as_uint(Bv.w)], true, vl);
            const float3 phi = beta * bsdf_f(vl, vf, xyz(Bv), wo, LB_ALL);
            atomicAdd(&L.flux[pix], make_float4(phi.x, phi.y, phi.z, 1.0f));
            deposits++;
        }
    }
    for (int off = 16; off > 0; off >>= 1) { deposits += __shfl_xor_sync(0xffffffffu, deposits, off); candidates += __shfl_xor_sync(0xffffffffu, candidates, off); }
    if (lane == 0 && deposits) atomicAdd(&L.stats[ST_DEPOSITS], (unsigned long long)deposits);
    if (lane == 0 && candidates) atomicAdd(&L.stats[ST_CANDIDATES], (unsigned long long)candidates);
}

// ---------------------------------------------------------------- per-iteration update and image (sppm.jl:438-472)
__global__ void __launch_bounds__(256) k_sppm_update(SppmLaunch L) {
    const float gamma = 2.0f / 3.0f;
    for (int pix = blockIdx.x * blockDim.x + threadIdx.x; pix < L.nstore; pix += gridDim.x * blockDim.x) {
        const float4 fl = L.flux[pix];
        if (fl.w > 0.0f) {
            float4 tr = L.tau_r[pix];
            const double N = L.N[pix];
            const double N_new = N + (double)(gamma * fl.w);
            const double radius_new = (double)tr.w * sqrt(N_new / (N + (double)fl.w));
            const double ratio = radius_new / (double)tr.w;
            const double r2 = ratio * ratio;
            tr.x = (float)((double)(tr.x + fl.x) * r2);
            tr.y = (float)((double)(tr.y + fl.y) * r2);
            tr.z = (float)((double)(tr.z + fl.z) * r2);
            tr.w = (float)radius_new;
            L.tau_r[pix] = tr;
            L.N[pix] = N_new;
            L.flux[pix] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        }
        L.vpC[pix].w = 0.0f;                                     // vp.beta = 0, vp.bsdf = nothing
    }
}

__global__ void __launch_bounds__(256) k_sppm_image(SppmLaunch L, int iteration, float* __restrict__ rgb) {
    const double Np = (double)iteration * (double)L.photons_per_iteration * 3.141592653589793;
    for (int pix = blockIdx.x * blockDim.x + threadIdx.x; pix < L.npix; pix += gridDim.x * blockDim.x) {
        const int st = raster_to_storage(L, pix % L.W, pix / L.W);
        const float4 ld = L.Ld[st], tr = L.tau_r[st];
        const double den = Np * (double)(tr.w * tr.w);
        rgb[3 * pix + 0] = ld.x / (float)iteration + (float)((double)tr.x / den);
        rgb[3 * pix + 1] = ld.y / (float)iteration + (float)((double)tr.y / den);
        rgb[3 * pix + 2] = ld.z / (float)iteration + (float)((double)tr.z / den);
    }
}

__global__ void k_sppm_init(SppmLaunch L, float r0) {
    for (int pix = blockIdx.x * blockDim.x + threadIdx.x; pix < L.nstore; pix += gridDim.x * blockDim.x) {
        L.Ld[pix] = make_float4(0, 0, 0, 0);
        L.flux[pix] = make_float4(0, 0, 0, 0);
        L.tau_r[pix] = make_float4(0, 0, 0, r0);
        L.N[pix] = 0.0;
        L.vpA[pix] = make_float4(0, 0, 0, 0); L.vpB[pix] = make_float4(0, 0, 0, 0); L.vpC[pix] = make_float4(0, 0, 0, 0);
        L.vpD[pix] = make_float4(0, 0, 0, 0); L.vpE[pix] = make_float4(0, 0, 0, 0);
    }
}

__global__ void k_sppm_stats(int* counters, unsigned long long* stats, int max_depth, int cap, int count_shadow) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        unsigned long long e = 0, s = 0;
        for (int l = 1; l <= max_depth; ++l) e += min(counters[l], cap);
        s = counters[32];
        atomicAdd(&stats[ST_RAYS_EXTEND], e);              // (lanes run concurrently)
        if (count_shadow) atomicAdd(&stats[ST_RAYS_SHADOW], s);      // in the photon pass slots 32.. count deposit requests
        else atomicAdd(&stats[ST_REQUESTS], s);
    }
}

// ---------------------------------------------------------------- host side
// Lanes: the camera pass and the photon pass are chains of ~12 dependent launches whose traversal launches cannot end
// before their slowest ray (0.2-0.5 ms in the 88k-triangle glass block, whatever the ray count).  Photon TRACING does
// not need the grid - only the deposits do - so it runs on its own streams concurrently with the camera pass, and each
// pass is cut into `K` sub-ranges on separate streams whose latency-bound tails overlap.
// Pipeline: the camera pass and the photon tracing of an iteration depend on nothing the previous iteration computes
// (paths are functions of (seed, pixel, iteration) / the Halton index; the radius enters only when the grid is built), so
// `D` iterations are in flight: iteration `it` uses slot (it - 1) % D - its own visible-point arrays, ray queues, request
// queue and streams - and only the chain grid -> deposit -> (all-reduce) -> update is serial on the main stream.  The
// latency-bound tails of one iteration's deep bounce levels (a traversal launch cannot end before its slowest ray) are
// filled by the next iteration's wide launches, and with a communicator the collectives overlap the next camera pass.
static const int SPPM_MAX_SLOTS = 8;
struct SppmState {
    SppmLaunch L;                   // slot 0's launch block (per-pixel state shared by all slots)
    SppmLaunch slotL[SPPM_MAX_SLOTS];
    int D = 1, cur_slot = 0;
    bool pipelined = false;         // set while sppm_iteration_async drives the passes (the stepwise API stays on slot 0)
    DevBuf vp_extra[SPPM_MAX_SLOTS][5];
    cudaEvent_t ev_slot_free[SPPM_MAX_SLOTS] = {};     // recorded on the main stream after the update that releases the slot
    DevBuf pix[10], grid, cells[4], scan_sums, q[10], pq[10], table, lights;
    float r0;
    int photon_cap;                 // photons one lane can hold
    int Kc = 1, Kp = 1;             // camera lanes use the context's lane ids 0..Kc-1, photon lanes Kc..Kc+Kp-1
    std::vector<SppmLaunch> cam_lane, ph_lane;
    cudaEvent_t ev_ph_fork = nullptr, ev_grid = nullptr;
    struct Traced { int it = -1; int64_t begin = 0, end = 0; } traced[SPPM_MAX_SLOTS];   // photon tracing already enqueued (per slot)
    cudaEvent_t ev_gathered[SPPM_MAX_SLOTS] = {};      // the slot's visible points are complete on this rank (all-gather done)
    cudaEvent_t ev_deposited = nullptr, ev_reduced = nullptr;
    bool active = false;
};

void sppm_free(trace_ctx* c) {                 // releases the device memory too (trace_destroy)
    if (!c->sppm) return;
    SppmState* s = c->sppm;
    for (auto& b : s->pix) b.release();
    for (auto& sl : s->vp_extra) for (auto& b : sl) b.release();
    for (auto& e : s->ev_slot_free) if (e) cudaEventDestroy(e);
    for (auto& e : s->ev_gathered) if (e) cudaEventDestroy(e);
    if (s->ev_deposited) cudaEventDestroy(s->ev_deposited);
    if (s->ev_reduced) cudaEventDestroy(s->ev_reduced);
    for (auto& b : s->cells) b.release();
    for (auto& b : s->q) b.release();
    for (auto& b : s->pq) b.release();
    if (s->ev_ph_fork) cudaEventDestroy(s->ev_ph_fork);
    if (s->ev_grid) cudaEventDestroy(s->ev_grid);
    s->grid.release(); s->scan_sums.release(); s->table.release(); s->lights.release();
    delete s;
    c->sppm = nullptr;
}
// ends a session but keeps the (grow-only) buffers: a caller rendering frame after frame (docs/code/caustic_moving.jl:
// 51 frames) does not pay ~1 GB of cudaMalloc / cudaFree per trace_render_sppm
void sppm_end_session(trace_ctx* c) {
    if (c->sppm) { c->sppm->active = false; for (auto& t : c->sppm->traced) t.it = -1; }
}

static float host_luminance_power(const trace_ctx*, const DeviceLight& l) {       // to_Y(power(light)), sppm.jl:564-569
    const float pi = 3.1415927f;
    float p[3];
    for (int k = 0; k < 3; ++k) {
        if (l.kind == TRACE_LIGHT_POINT) p[k] = (4.0f * pi) * l.I[k];
        else p[k] = ((l.I[k] * 2.0f) * pi) * (1.0f - 0.5f * (l.cos_falloff + l.cos_total));
    }
    return (0.212671f * p[0] + 0.715160f * p[1]) + 0.072169f * p[2];
}

extern "C" int trace_sppm_begin(trace_ctx* c, const trace_camera* cam, const trace_film_desc* film, float r0, int max_depth,
                                int64_t photons, uint64_t seed) {
    if (!c) return 1;
    cudaSetDevice(c->device);
    if (!c->have_scene) return c->fail("no scene uploaded");
    if (!cam || !film) return c->fail("trace_sppm_begin: null argument");
    if (max_depth < 1 || max_depth > TR_MAX_DEPTH) return c->fail("trace_sppm_begin: max_depth must be in [1, %d]", TR_MAX_DEPTH);
    if (!(r0 > 0.0f)) return c->fail("trace_sppm_begin: bad radius");
    if (c->scene.n_lights < 1) return c->fail("trace_sppm_begin: the scene has no lights");
    sppm_end_session(c);
    if (!c->sppm) c->sppm = new SppmState();
    SppmState* s = c->sppm;
    SppmLaunch& L = s->L;
    memset(&L, 0, sizeof(L));
    L.sc = c->scene;
    ctx_device_camera(cam, &L.cam);
    if (ctx_device_film(c, film, &L.film, &s->table)) return 1;
    L.W = L.film.width; L.H = L.film.height; L.npix = L.W * L.H;
    {   // grid_hash's division-free modulo
        int lg = 0;
        while ((1ull << lg) < (unsigned long long)L.npix) ++lg;
        const int k = 57 + lg;
        L.hash_shift = k - 64;
        L.hash_magic = 0;
        if (L.hash_shift >= 0) {
            const unsigned __int128 one = (unsigned __int128)1 << k;
            L.hash_magic = (unsigned long long)((one + (unsigned __int128)L.npix - 1) / (unsigned __int128)L.npix);
        }
    }
    if (c->rank < 0 || c->rank >= c->world) return c->fail("rank %d outside world %d", c->rank, c->world);
    L.world = c->world; L.rank = c->rank;
    L.chunk_rows = (L.H + L.world - 1) / L.world;
    L.nstore = L.world * L.chunk_rows * L.W;
    if (photons <= 0) photons = (int64_t)(film->crop_x1 - film->crop_x0) * (film->crop_y1 - film->crop_y0);   // area(crop_bounds), Q22
    L.photons_per_iteration = photons;
    L.max_depth = max_depth; L.seed = seed; L.iteration = 0;
    s->r0 = r0;
    const size_t np = (size_t)L.nstore;
    const size_t f4b = np * sizeof(float4);
    for (int k = 0; k < 8; ++k) TR_CUDA(c, s->pix[k].ensure(f4b));
    TR_CUDA(c, s->pix[8].ensure(np * sizeof(double)));
    L.Ld = s->pix[0].as<float4>(); L.flux = s->pix[1].as<float4>(); L.tau_r = s->pix[2].as<float4>();
    L.vpA = s->pix[3].as<float4>(); L.vpB = s->pix[4].as<float4>(); L.vpC = s->pix[5].as<float4>();
    L.vpD = s->pix[6].as<float4>(); L.vpE = s->pix[7].as<float4>(); L.N = s->pix[8].as<double>();
    TR_CUDA(c, s->grid.ensure(sizeof(GridParams)));
    L.grid = s->grid.as<GridParams>();
    L.items_cap = (unsigned int)std::min<size_t>(np * 28 + 1024, 0xFFFFFF00u);
    TR_CUDA(c, s->cells[0].ensure((np + 1) * sizeof(unsigned int)));
    TR_CUDA(c, s->cells[1].ensure((np + 1) * sizeof(unsigned int)));
    TR_CUDA(c, s->cells[2].ensure((size_t)L.items_cap * sizeof(unsigned int)));
    TR_CUDA(c, s->cells[3].ensure((size_t)L.items_cap * sizeof(float4)));
    L.cell_vp = s->cells[3].as<float4>();
    L.cell_start = s->cells[0].as<unsigned int>(); L.cell_cursor = s->cells[1].as<unsigned int>();
    L.cell_items = s->cells[2].as<unsigned int>();
    const int scan_blocks = (int)((np + 1 + SCAN_BLOCK * SCAN_ITEMS - 1) / (SCAN_BLOCK * SCAN_ITEMS));
    TR_CUDA(c, s->scan_sums.ensure((size_t)scan_blocks * sizeof(unsigned int)));
    // one camera lane + one photon lane by default: measured on B200, cutting the passes further (sppm_lanes 2/4/8) only
    // adds launches - the traversal launches of these scenes are throughput-bound (the glass block's degenerate BVH
    // costs every ray ~1000 node visits), not bound by a few slow rays (profiles/r1_experiments.md)
    const int K = c->sppm_lanes > 0 ? c->sppm_lanes : 1;
    s->Kc = s->Kp = std::min(K, trace_ctx::MAX_LANES / 2);
    // iterations in flight (see SppmState): every slot needs Kc + Kp lanes (streams, counter blocks)
    s->D = std::max(1, std::min(std::min(c->sppm_pipeline, SPPM_MAX_SLOTS), trace_ctx::MAX_LANES / (s->Kc + s->Kp)));
    s->cur_slot = 0; s->pipelined = false;
    for (int d = 0; d < s->D; ++d) {
        if (!s->ev_slot_free[d]) TR_CUDA(c, cudaEventCreateWithFlags(&s->ev_slot_free[d], cudaEventDisableTiming));
        if (!s->ev_gathered[d]) TR_CUDA(c, cudaEventCreateWithFlags(&s->ev_gathered[d], cudaEventDisableTiming));
    }
    if (!s->ev_deposited) TR_CUDA(c, cudaEventCreateWithFlags(&s->ev_deposited, cudaEventDisableTiming));
    if (!s->ev_reduced) TR_CUDA(c, cudaEventCreateWithFlags(&s->ev_reduced, cudaEventDisableTiming));
    for (int d = 1; d < s->D; ++d)
        for (int k = 0; k < 5; ++k) {
            TR_CUDA(c, s->vp_extra[d][k].ensure(f4b));
            TR_CUDA(c, cudaMemsetAsync(s->vp_extra[d][k].p, 0, f4b, c->stream));
        }
    if (!s->ev_ph_fork) TR_CUDA(c, cudaEventCreateWithFlags(&s->ev_ph_fork, cudaEventDisableTiming));
    if (!s->ev_grid) TR_CUDA(c, cudaEventCreateWithFlags(&s->ev_grid, cudaEventDisableTiming));
    // camera queues hold this rank's pixels, photon queues one chunk of photons; both are cut evenly over the lanes
    const size_t rank_slots = (size_t)L.chunk_rows * L.W;
    const size_t cam_cap = (rank_slots + s->Kc - 1) / s->Kc;
    const size_t ph_total = (size_t)std::min<int64_t>(photons, std::max<int64_t>(c->batch * 2, 1 << 20));
    const size_t ph_cap = (ph_total + s->Kp - 1) / s->Kp;
    s->photon_cap = (int)ph_cap;
    L.counters = ctx_icounters_lane(c, 0);
    L.flags = ctx_icounters_lane(c, 0);
    L.stats = ctx_stats64(c);
    L.cap = 0; L.cap_shadow = 0; L.range_begin = L.range_end = 0;
    // lanes of all slots: lane index = slot * K_ + sub-range
    auto carve = [&](DevBuf* q, int K_, size_t cap, std::vector<SppmLaunch>& lanes, int lane0) -> int {
        const size_t cap_sh = std::min<size_t>(cap * (size_t)max_depth, (size_t)1 << 30);
        const int n_lanes = s->D * K_;
        for (int k = 0; k < 7; ++k) TR_CUDA(c, q[k].ensure((size_t)n_lanes * cap * sizeof(float4)));
        for (int k = 7; k < 10; ++k) TR_CUDA(c, q[k].ensure((size_t)n_lanes * cap_sh * sizeof(float4)));
        lanes.resize((size_t)n_lanes);
        for (int l = 0; l < n_lanes; ++l) {
            lanes[l] = s->slotL[l / K_];
            SppmLaunch& W = lanes[l];
            W.ro[0] = q[0].as<float4>() + l * cap; W.ro[1] = q[1].as<float4>() + l * cap;
            W.rd[0] = q[2].as<float4>() + l * cap; W.rd[1] = q[3].as<float4>() + l * cap;
            W.rw[0] = q[4].as<float4>() + l * cap; W.rw[1] = q[5].as<float4>() + l * cap;
            W.hits = q[6].as<float4>() + l * cap;
            W.so = q[7].as<float4>() + l * cap_sh; W.sd = q[8].as<float4>() + l * cap_sh; W.sc_contrib = q[9].as<float4>() + l * cap_sh;
            W.cap = (int)cap; W.cap_shadow = (int)cap_sh;
            W.counters = ctx_icounters_lane(c, lane0 + l);
        }
        return 0;
    };
    // (lanes are carved again below, once the light tables are in L)
    // light power distribution: Distribution1D (sampling.jl:3-30), built on the host from the uploaded lights
    const int nl = c->scene.n_lights;
    std::vector<DeviceLight> hl((size_t)nl);
    TR_CUDA(c, cudaMemcpyAsync(hl.data(), c->scene.lights, (size_t)nl * sizeof(DeviceLight), cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(c, cudaStreamSynchronize(c->stream));
    std::vector<float> func((size_t)nl), cdf((size_t)nl + 1);
    for (int i = 0; i < nl; ++i) {
        // the reference defines no sample_le for DirectionalLight (lights/directional.jl): its photon pass would throw
        if (hl[i].kind == TRACE_LIGHT_DIRECTIONAL) { return c->fail("SPPM: DirectionalLight cannot emit photons (no sample_le in the reference)"); }
        func[i] = host_luminance_power(c, hl[i]);
    }
    cdf[0] = 0.0f;
    for (int i = 1; i <= nl; ++i) cdf[i] = cdf[i - 1] + func[i - 1] / (float)nl;
    const float func_int = cdf[nl];
    if (func_int == 0.0f) { for (int i = 1; i <= nl; ++i) cdf[i] = (float)(i + 1) / (float)nl; }
    else { for (int i = 1; i <= nl; ++i) cdf[i] /= func_int; }
    std::vector<float> pack(cdf);
    pack.insert(pack.end(), func.begin(), func.end());
    TR_CUDA(c, s->lights.ensure(pack.size() * sizeof(float)));
    TR_CUDA(c, cudaMemcpyAsync(s->lights.p, pack.data(), pack.size() * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    TR_CUDA(c, cudaStreamSynchronize(c->stream));
    L.light_cdf = s->lights.as<float>(); L.light_func = s->lights.as<float>() + nl + 1; L.light_func_int = func_int;
    for (int d = 0; d < s->D; ++d) {
        s->slotL[d] = L;
        if (d > 0) {
            SppmLaunch& S = s->slotL[d];
            S.vpA = s->vp_extra[d][0].as<float4>(); S.vpB = s->vp_extra[d][1].as<float4>(); S.vpC = s->vp_extra[d][2].as<float4>();
            S.vpD = s->vp_extra[d][3].as<float4>(); S.vpE = s->vp_extra[d][4].as<float4>();
        }
    }
    if (carve(s->q, s->Kc, cam_cap, s->cam_lane, 0) || carve(s->pq, s->Kp, ph_cap, s->ph_lane, s->D * s->Kc)) return 1;
    for (int l = 0; l < s->D * s->Kc; ++l) {
        const size_t s0 = (size_t)L.rank * rank_slots;
        const int sub = l % s->Kc;
        s->cam_lane[l].range_begin = (int)(s0 + std::min(rank_slots, (size_t)sub * cam_cap));
        s->cam_lane[l].range_end = (int)(s0 + std::min(rank_slots, (size_t)(sub + 1) * cam_cap));
    }
    k_sppm_init<<<persistent_grid(c, 4), 256, 0, c->stream>>>(L, r0);
    c->stats.kernel_launches++;
    TR_CUDA(c, cudaGetLastError());
    for (int d = 0; d < s->D; ++d) TR_CUDA(c, cudaEventRecord(s->ev_slot_free[d], c->stream));      // every slot starts out free
    s->active = true;
    return 0;
}

static int check_flags(trace_ctx* c, const char* what) {
    int* ic = ctx_icounters(c);
    TR_CUDA(c, cudaMemcpyAsync(c->h_flags, ic + IC_OVERFLOW, 4 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(c, cudaStreamSynchronize(c->stream));
    c->kev_collect();
    if (c->h_flags[0] | c->h_flags[1] | c->h_flags[2] | c->h_flags[3]) cudaMemsetAsync(ic + IC_OVERFLOW, 0, 4 * sizeof(int), c->stream);
    if (c->h_flags[1]) return c->fail("%s: traversal stack overflow (> 64 pending nodes)", what);
    if (c->h_flags[0]) return c->fail("%s: SPPM grid item capacity exceeded (more than 28 grid cells per visible point on average)", what);
    if (c->h_flags[2]) return c->fail("%s: SPPM shadow-ray queue overflow (direct-lighting samples of the camera pass were dropped)", what);
    if (c->h_flags[3]) return c->fail("%s: SPPM deposit-request queue overflow (photon deposits were dropped)", what);
    return 0;
}

// Runs `body(lane)` for every lane on its own side stream (forked from / joined into the main stream), or directly on
// the main stream when there is only one lane and `fork_event` is null.
struct LaneScope {
    trace_ctx* c;
    LaneScope(trace_ctx* c_, int lane, cudaStream_t st) : c(c_) { c->cur_lane = lane; c->cur_stream = st; }
    ~LaneScope() { c->cur_lane = 0; c->cur_stream = c->stream; }
};

static int sppm_camera_lane(trace_ctx* c, SppmState* s, int l, int iteration) {
    TrRange nvtx("sppm.camera pass");
    SppmLaunch& W = s->cam_lane[l];
    W.iteration = iteration;
    cudaStream_t st = c->cur_stream;
    int* ic = W.counters;
    unsigned long long* stats = ctx_stats64(c);
    TR_CUDA(c, cudaMemsetAsync(ic, 0, 60 * sizeof(int), st));
    TR_CUDA(c, cudaMemsetAsync(ic + 64, 0, 64 * sizeof(int), st)); c->work_slot = 0;
    const int g_stream = persistent_grid(c, 8), g_trav = persistent_grid(c, 16);
    const bool path = c->sppm_path && c->slab != 1;
    if (path) {
        // all bounce levels of the camera paths in ONE launch (k_sppm_cam_path); rays are counted by the kernel itself
        c->kev_begin(TRACE_K_EXTEND);
        trav_dispatch(c, [&](auto S, auto C_, auto Wk) {
            constexpr int s_ = decltype(S)::value, w_ = decltype(Wk)::value;
            constexpr bool cn = decltype(C_)::value;
            SppmLaunch P = W;
            P.sc = hit_launch_scene(c, W.sc);
            auto k = k_sppm_cam_path<s_, cn, w_, false>;
            if constexpr (shadow_walk_capable<s_, cn, w_>) if (P.sc.shadow_pairs) k = k_sppm_cam_path<s_, cn, w_, true>;
            k<<<occupancy_grid(c, k, 128), 128, 0, st>>>(P, c->sppm_path, W.flags + IC_ERROR);
        });
        c->kev_end();
        c->stats.kernel_launches++;
        for (int level = c->sppm_path + 1; level <= W.max_depth; ++level) {
            const int cur = (level - 1) & 1;
            c->cur_level = level;
            launch_extend(c, g_trav, W.sc, (const float4*)W.ro[cur], (const float4*)W.rd[cur], (const int*)(ic + level), W.cap, W.hits,
                          stats + ST_NODES, W.flags + IC_ERROR);
            c->kev_begin(TRACE_K_SHADE);
            k_sppm_cam_shade<<<occupancy_grid(c, k_sppm_cam_shade, 128), 128, 0, st>>>(W, level);
            c->kev_end();
            c->stats.kernel_launches++;
        }
    } else {
        c->kev_begin(TRACE_K_GENERATE);
        k_sppm_cam_generate<<<g_stream, 256, 0, st>>>(W);
        c->kev_end();
        c->stats.kernel_launches++;
        for (int level = 1; level <= W.max_depth; ++level) {
            const int cur = (level - 1) & 1;
            c->cur_level = level;
            launch_extend(c, g_trav, W.sc, (const float4*)W.ro[cur], (const float4*)W.rd[cur], (const int*)(ic + level), W.cap, W.hits,
                          stats + ST_NODES, W.flags + IC_ERROR);
            c->kev_begin(TRACE_K_SHADE);
            k_sppm_cam_shade<<<occupancy_grid(c, k_sppm_cam_shade, 128), 128, 0, st>>>(W, level);
            c->kev_end();
            c->stats.kernel_launches++;
        }
    }
    // shadow rays of all levels in one any-hit launch (they only feed Ld)
    launch_shadow(c, g_trav, W.sc, (const float4*)W.so, (const float4*)W.sd, (const float4*)W.sc_contrib,
                  (const int*)(ic + 32), W.cap_shadow, W.Ld, stats + ST_NODES, W.flags + IC_ERROR);
    k_sppm_stats<<<1, 32, 0, st>>>(ic, stats, W.max_depth, W.cap, 1);      // (levels run by the path kernel have counter 0: it counts its own rays)
    c->stats.kernel_launches++;
    return 0;
}

// camera pass of this rank's rows, enqueued only (no host wait)
// `join` false: the caller makes whoever needs the visible points wait for the slot's lanes (sppm_join_camera)
static int sppm_camera_pass_async(trace_ctx* c, int iteration, bool join = true) {
    if (!c) return 1;
    cudaSetDevice(c->device);
    if (!c->sppm || !c->sppm->active) return c->fail("trace_sppm_camera_pass: call trace_sppm_begin first");
    SppmState* s = c->sppm;
    s->L.iteration = iteration;
    // the slot's lanes wait only until the update that last used the slot's visible-point arrays has run
    // (D iterations back); the main stream then waits for them: everything after this call sees the visible points
    const int slot = s->pipelined ? (iteration - 1) % s->D : 0;
    s->cur_slot = slot;
    s->slotL[slot].iteration = iteration;
    for (int l = 0; l < s->Kc; ++l) {
        const int lane = slot * s->Kc + l;
        TR_CUDA(c, cudaStreamWaitEvent(c->side[lane], s->ev_slot_free[slot], 0));
        LaneScope scope(c, lane, c->side[lane]);
        if (sppm_camera_lane(c, s, lane, iteration)) return 1;
        TR_CUDA(c, cudaEventRecord(c->ev_join[lane], c->side[lane]));
        if (join) TR_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_join[lane], 0));
    }
    TR_CUDA(c, cudaGetLastError());
    return 0;
}
static int sppm_join_camera(trace_ctx* c, int slot, cudaStream_t waiter) {
    SppmState* s = c->sppm;
    for (int l = 0; l < s->Kc; ++l) TR_CUDA(c, cudaStreamWaitEvent(waiter, c->ev_join[slot * s->Kc + l], 0));
    return 0;
}

static int sppm_build_grid_async(trace_ctx* c);

extern "C" int trace_sppm_camera_pass(trace_ctx* c, int iteration) {
    if (sppm_camera_pass_async(c, iteration, true)) return 1;
    if (c->world > 1) return check_flags(c, "trace_sppm_camera_pass");   // caller all-gathers the visible points, then build_grid
    return trace_sppm_build_grid(c);
}

// hash grid of the visible points (sppm.jl:272-318): bounds -> resolution -> count -> scan -> fill
extern "C" int trace_sppm_build_grid(trace_ctx* c) {
    if (sppm_build_grid_async(c)) return 1;
    return check_flags(c, "trace_sppm_build_grid");
}
static int sppm_build_grid_async(trace_ctx* c) {
    TrRange nvtx("sppm.grid build");
    if (!c) return 1;
    cudaSetDevice(c->device);
    if (!c->sppm || !c->sppm->active) return c->fail("trace_sppm_build_grid: call trace_sppm_begin first");
    SppmState* s = c->sppm;
    SppmLaunch& L = s->slotL[s->cur_slot];
    const int g_stream = persistent_grid(c, 8);
    const int n_cells = L.npix + 1;
    const int scan_blocks = (n_cells + SCAN_BLOCK * SCAN_ITEMS - 1) / (SCAN_BLOCK * SCAN_ITEMS);
    c->kev_begin(TRACE_K_GRID);                                 // (the ten launches of the grid build are timed as one)
    k_grid_reset<<<1, 1, 0, c->stream>>>(L.grid);
    k_grid_bounds<<<g_stream, 256, 0, c->stream>>>(L);
    k_grid_params<<<1, 1, 0, c->stream>>>(L.grid);
    TR_CUDA(c, cudaMemsetAsync(L.cell_start, 0, (size_t)n_cells * sizeof(unsigned int), c->stream));
    k_grid_insert<false><<<g_stream, 256, 0, c->stream>>>(L);
    k_scan_blocks<<<scan_blocks, SCAN_BLOCK, 0, c->stream>>>(L.cell_start, n_cells, s->scan_sums.as<unsigned int>());
    k_scan_sums<<<1, 32, 0, c->stream>>>(s->scan_sums.as<unsigned int>(), scan_blocks, L.grid);
    k_scan_add<<<scan_blocks, SCAN_BLOCK, 0, c->stream>>>(L.cell_start, n_cells, s->scan_sums.as<unsigned int>(), L.cell_cursor);
    k_grid_check<<<1, 1, 0, c->stream>>>(L);
    k_grid_insert<true><<<g_stream, 256, 0, c->stream>>>(L);
    c->kev_end();
    c->stats.kernel_launches += 10;
    TR_CUDA(c, cudaGetLastError());
    return 0;
}

// Photon tracing of [begin, end) on the photon lanes: generate -> (extend -> shade) x depth.  The shade kernel leaves
// deposit REQUESTS (hit point, direction, weight) in the lane's request queue; nothing here reads the grid.
static int sppm_trace_lane(trace_ctx* c, SppmState* s, int j, int iteration, int64_t b, int n) {
    TrRange nvtx("sppm.photon tracing");
    SppmLaunch& W = s->ph_lane[j];
    W.iteration = iteration;
    W.photon_begin = b;
    W.n_photons = n;
    cudaStream_t st = c->cur_stream;
    int* ic = W.counters;
    unsigned long long* stats = ctx_stats64(c);
    TR_CUDA(c, cudaMemsetAsync(ic, 0, 60 * sizeof(int), st));
    TR_CUDA(c, cudaMemsetAsync(ic + 64, 0, 64 * sizeof(int), st)); c->work_slot = 0;
    const int g_stream = persistent_grid(c, 8), g_trav = persistent_grid(c, 16);
    if (c->sppm_path && c->slab != 1) {
        c->kev_begin(TRACE_K_EXTEND);
        trav_dispatch(c, [&](auto S, auto C_, auto Wk) {
            constexpr int s_ = decltype(S)::value, w_ = decltype(Wk)::value;
            constexpr bool cn = decltype(C_)::value;
            SppmLaunch P = W;
            P.sc = hit_launch_scene(c, W.sc);
            auto k = k_photon_path<s_, cn, w_, false>;
            if constexpr (shadow_walk_capable<s_, cn, w_>) if (P.sc.shadow_pairs) k = k_photon_path<s_, cn, w_, true>;
            k<<<occupancy_grid(c, k, 128), 128, 0, st>>>(P, c->sppm_path, W.flags + IC_ERROR);
        });
        c->kev_end();
        c->stats.kernel_launches++;
        for (int level = c->sppm_path + 1; level <= W.max_depth; ++level) {
            const int cur = (level - 1) & 1;
            c->cur_level = level;
            launch_extend(c, g_trav, W.sc, (const float4*)W.ro[cur], (const float4*)W.rd[cur], (const int*)(ic + level), W.cap, W.hits,
                          stats + ST_NODES, W.flags + IC_ERROR);
            c->kev_begin(TRACE_K_SHADE);
            k_photon_shade<<<occupancy_grid(c, k_photon_shade, 128), 128, 0, st>>>(W, level);
            c->kev_end();
            c->stats.kernel_launches++;
        }
        return 0;
    }
    c->kev_begin(TRACE_K_GENERATE);
    k_photon_generate<<<g_stream, 256, 0, st>>>(W);
    c->kev_end();
    c->stats.kernel_launches++;
    for (int level = 1; level <= W.max_depth; ++level) {
        const int cur = (level - 1) & 1;
        c->cur_level = level;
        launch_extend(c, g_trav, W.sc, (const float4*)W.ro[cur], (const float4*)W.rd[cur], (const int*)(ic + level), W.cap, W.hits,
                      stats + ST_NODES, W.flags + IC_ERROR);
        c->kev_begin(TRACE_K_SHADE);
        k_photon_shade<<<occupancy_grid(c, k_photon_shade, 128), 128, 0, st>>>(W, level);
        c->kev_end();
        c->stats.kernel_launches++;
    }
    return 0;
}

static int sppm_deposit_lane(trace_ctx* c, SppmState* s, int j) {
    TrRange nvtx("sppm.photon deposit");
    SppmLaunch& W = s->ph_lane[j];
    cudaStream_t st = c->cur_stream;
    // deposit requests of all bounce levels in one launch (deposits do not feed back into the photon paths)
    c->kev_begin(TRACE_K_DEPOSIT);
    k_photon_deposit<<<occupancy_grid(c, k_photon_deposit, 128), 128, 0, st>>>(W, 0);
    c->kev_end();
    k_sppm_stats<<<1, 32, 0, st>>>(W.counters, ctx_stats64(c), W.max_depth, W.cap, 0);
    c->stats.kernel_launches += 2;
    return 0;
}

// Starts tracing this iteration's photons [begin, end) WITHOUT depositing them.  Call it before trace_sppm_camera_pass:
// the photon paths then run concurrently with the camera pass (and with the caller's all-gather of the visible points);
// trace_sppm_photon_pass(iteration, begin, end) later only joins and deposits.  Optional: photon_pass traces by itself
// when this was not called (or the range does not fit the photon queues in one go).
extern "C" int trace_sppm_trace_photons(trace_ctx* c, int iteration, int64_t begin, int64_t end) {
    if (!c) return 1;
    cudaSetDevice(c->device);
    if (!c->sppm || !c->sppm->active) return c->fail("trace_sppm_trace_photons: call trace_sppm_begin first");
    SppmState* s = c->sppm;
    if (begin < 0 || end > s->L.photons_per_iteration || begin > end) return c->fail("trace_sppm_trace_photons: bad photon range");
    const int tslot = s->pipelined ? (iteration - 1) % s->D : 0;
    s->traced[tslot].it = -1;
    if (end - begin > (int64_t)s->photon_cap * s->Kp) return 0;          // does not fit: photon_pass will chunk it
    const int64_t per = (end - begin + s->Kp - 1) / s->Kp;
    // Photon paths read nothing an earlier iteration writes; the lane's own stream orders them after the deposits that
    // last read its request queue (D iterations back).  Only a session's first use of a lane waits for the main stream.
    const int slot = s->pipelined ? (iteration - 1) % s->D : 0;
    const bool first_use = iteration <= (s->pipelined ? s->D : 1);
    if (first_use) TR_CUDA(c, cudaEventRecord(s->ev_ph_fork, c->stream));
    for (int j = 0; j < s->Kp; ++j) {
        const int idx = slot * s->Kp + j, lane = s->D * s->Kc + idx;
        const int64_t b = std::min(end, begin + j * per), e = std::min(end, b + per);
        if (first_use) TR_CUDA(c, cudaStreamWaitEvent(c->side[lane], s->ev_ph_fork, 0));
        LaneScope scope(c, lane, c->side[lane]);
        if (sppm_trace_lane(c, s, idx, iteration, b, (int)(e - b))) return 1;
    }
    TR_CUDA(c, cudaGetLastError());
    s->traced[tslot].it = iteration; s->traced[tslot].begin = begin; s->traced[tslot].end = end;
    return 0;
}

extern "C" int trace_sppm_photon_pass(trace_ctx* c, int iteration, int64_t begin, int64_t end) {
    if (!c) return 1;
    cudaSetDevice(c->device);
    if (!c->sppm || !c->sppm->active) return c->fail("trace_sppm_photon_pass: call trace_sppm_begin first");
    SppmState* s = c->sppm;
    if (begin < 0 || end > s->L.photons_per_iteration || begin > end) return c->fail("trace_sppm_photon_pass: bad photon range");
    s->L.iteration = iteration;
    const int64_t chunk = (int64_t)s->photon_cap * s->Kp;
    for (int64_t b0 = begin;; b0 += chunk) {
        const int64_t e0 = std::min(end, b0 + chunk);
        SppmState::Traced& tr = s->traced[s->pipelined ? (iteration - 1) % s->D : 0];
        if (!(tr.it == iteration && tr.begin == b0 && tr.end == e0))
            if (trace_sppm_trace_photons(c, iteration, b0, e0)) return 1;
        tr.it = -1;
        // the deposits need the grid (main stream): every photon lane waits for it, deposits, and joins the main stream
        TR_CUDA(c, cudaEventRecord(s->ev_grid, c->stream));
        const int slot = s->pipelined ? (iteration - 1) % s->D : 0;
        for (int j = 0; j < s->Kp; ++j) {
            const int idx = slot * s->Kp + j, lane = s->D * s->Kc + idx;
            TR_CUDA(c, cudaStreamWaitEvent(c->side[lane], s->ev_grid, 0));
            LaneScope scope(c, lane, c->side[lane]);
            if (sppm_deposit_lane(c, s, idx)) return 1;
            TR_CUDA(c, cudaEventRecord(c->ev_join[lane], c->side[lane]));
            TR_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_join[lane], 0));
        }
        if (e0 >= end) break;
    }
    TR_CUDA(c, cudaGetLastError());
    return 0;
}

extern "C" void* trace_sppm_flux_device(trace_ctx* c, int64_t* n_floats) { return trace_sppm_buffer_device(c, 0, n_floats); }

// Per-pixel device buffers in STORAGE order (rank r owns the contiguous slice [r, r+1) * n_floats / world):
// 0 flux (Phi.rgb, M) - all-reduce(sum) after the photon pass; 1 Ld - all-gather before the image;
// 2..6 visible-point records - all-gather after the camera pass.
extern "C" void* trace_sppm_buffer_device(trace_ctx* c, int which, int64_t* n_floats) {
    if (!c || !c->sppm) return nullptr;
    SppmLaunch& L = c->sppm->L;
    if (n_floats) *n_floats = (int64_t)L.nstore * 4;
    switch (which) {
        case 0: return L.flux;
        case 1: return L.Ld;
        case 2: return L.vpA;
        case 3: return L.vpB;
        case 4: return L.vpC;
        case 5: return L.vpD;
        case 6: return L.vpE;
        default: return nullptr;
    }
}

extern "C" int trace_sppm_update(trace_ctx* c) {
    if (!c) return 1;
    cudaSetDevice(c->device);
    if (!c->sppm || !c->sppm->active) return c->fail("trace_sppm_update: call trace_sppm_begin first");
    SppmState* s = c->sppm;
    c->kev_begin(TRACE_K_UPDATE);
    k_sppm_update<<<persistent_grid(c, 4), 256, 0, c->stream>>>(s->slotL[s->cur_slot]);
    c->kev_end();
    c->stats.kernel_launches++;
    TR_CUDA(c, cudaGetLastError());
    TR_CUDA(c, cudaEventRecord(s->ev_slot_free[s->cur_slot], c->stream));     // the slot's visible-point arrays may be overwritten
    return 0;
}

extern "C" int trace_sppm_image(trace_ctx* c, int iteration, float* rgb_out) {
    if (!c) return 1;
    cudaSetDevice(c->device);
    if (!c->sppm || !c->sppm->active) return c->fail("trace_sppm_image: call trace_sppm_begin first");
    if (!rgb_out || iteration < 1) return c->fail("trace_sppm_image: bad argument");
    SppmLaunch& L = c->sppm->L;
    const size_t bytes = (size_t)L.npix * 3 * sizeof(float);
    TR_CUDA(c, c->b_misc[6].ensure(bytes));
    if (c->comm && c->world > 1) {       // Ld is accumulated only by the rank that owns the row: gather it (idempotent)
        const size_t slice = (size_t)L.nstore / (size_t)c->world * 4;
        float* base = reinterpret_cast<float*>(L.Ld);
        if (comm_allgather(c, base + (size_t)c->rank * slice, base, slice)) return 1;
    }
    k_sppm_image<<<persistent_grid(c, 4), 256, 0, c->stream>>>(L, iteration, c->b_misc[6].as<float>());
    c->stats.kernel_launches++;
    TR_CUDA(c, cudaMemcpyAsync(rgb_out, c->b_misc[6].p, bytes, cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(c, cudaStreamSynchronize(c->stream));
    return check_flags(c, "trace_sppm_image");
}

extern "C" int trace_sppm_end(trace_ctx* c) {
    if (!c) return 1;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    sppm_end_session(c);
    return 0;
}

// SPPM iterations (sppm.jl:153-165) enqueued on the context's streams without any host wait.  An iteration is two phases:
//   A  photon tracing + camera pass on the slot's own streams, and - with a communicator - the all-gather of the
//      visible points (camera paths are sharded by image rows) on the COLLECTIVE stream;
//   B  the serial chain on the main stream: hash grid -> deposits -> all-reduce(sum) of (Phi, M) (photons are sharded by
//      index range; collective stream) -> update.
// Phase A of iteration it + 1 is enqueued BEFORE phase B of iteration it: NCCL runs a communicator's operations in
// issue order, so the next all-gather then sits in front of this iteration's all-reduce and overlaps the chain instead of
// extending it (measured on 8 B200, caustic_moving: the chain - all-gather 0.25 + grid 0.33 + deposits 0.1 + all-reduce
// 0.25 ms - was the whole iteration).  Needs two slots (the look-ahead pass must not reuse the slot in flight).
static int sppm_phase_a(trace_ctx* c, int it) {
    SppmState* s = c->sppm;
    SppmLaunch& L = s->L;
    const bool multi = c->comm != nullptr && c->world > 1;
    const int64_t P = L.photons_per_iteration;
    const int64_t b = multi ? P * c->rank / c->world : 0, e = multi ? P * (c->rank + 1) / c->world : P;
    // photon tracing first: it does not need the grid and overlaps the camera pass (and the all-gather) on its own stream
    if (trace_sppm_trace_photons(c, it, b, e) || sppm_camera_pass_async(c, it, false)) return 1;
    const int slot = s->cur_slot;
    if (!multi) return 0;
    // rank r owns slice r of every per-pixel array (storage order): five in-place all-gathers, one NCCL launch
    if (sppm_join_camera(c, slot, c->coll_stream)) return 1;
    const size_t slice = (size_t)L.nstore / (size_t)c->world * 4;
    const SppmLaunch& S = s->slotL[slot];
    float4* arr[5] = {S.vpA, S.vpB, S.vpC, S.vpD, S.vpE};
    struct CollScope {
        trace_ctx* c; cudaStream_t saved, saved_cur;
        explicit CollScope(trace_ctx* c_) : c(c_), saved(c_->stream), saved_cur(c_->cur_stream) { c->stream = c->cur_stream = c->coll_stream; }
        ~CollScope() { c->stream = saved; c->cur_stream = saved_cur; }
    } coll(c);
    c->kev_begin(TRACE_K_COMM);
    if (comm_group_begin(c)) return 1;
    for (int k = 0; k < 5; ++k) {
        float* base = reinterpret_cast<float*>(arr[k]);
        if (comm_allgather(c, base + (size_t)c->rank * slice, base, slice)) { comm_group_end(c); return 1; }
    }
    if (comm_group_end(c)) return 1;
    c->kev_end();
    TR_CUDA(c, cudaEventRecord(s->ev_gathered[slot], c->coll_stream));
    return 0;
}

static int sppm_phase_b(trace_ctx* c, int it) {
    SppmState* s = c->sppm;
    SppmLaunch& L = s->L;
    const bool multi = c->comm != nullptr && c->world > 1;
    const int64_t P = L.photons_per_iteration;
    const int64_t b = multi ? P * c->rank / c->world : 0, e = multi ? P * (c->rank + 1) / c->world : P;
    const int slot = (it - 1) % s->D;
    s->cur_slot = slot;                                          // (phase A of the next iteration moved it on)
    if (multi) TR_CUDA(c, cudaStreamWaitEvent(c->stream, s->ev_gathered[slot], 0));
    else if (sppm_join_camera(c, slot, c->stream)) return 1;
    if (sppm_build_grid_async(c) || trace_sppm_photon_pass(c, it, b, e)) return 1;
    if (multi) {
        TR_CUDA(c, cudaEventRecord(s->ev_deposited, c->stream));
        TR_CUDA(c, cudaStreamWaitEvent(c->coll_stream, s->ev_deposited, 0));
        {
            cudaStream_t saved = c->stream, saved_cur = c->cur_stream;
            c->stream = c->cur_stream = c->coll_stream;
            c->kev_begin(TRACE_K_COMM);
            const int rc = comm_allreduce_sum(c, reinterpret_cast<float*>(L.flux), (size_t)L.nstore * 4);
            c->kev_end();
            c->stream = saved; c->cur_stream = saved_cur;
            if (rc) return 1;
        }
        TR_CUDA(c, cudaEventRecord(s->ev_reduced, c->coll_stream));
        TR_CUDA(c, cudaStreamWaitEvent(c->stream, s->ev_reduced, 0));
    }
    return trace_sppm_update(c);
}

// iterations first .. first + n - 1
static int sppm_iterations_async(trace_ctx* c, int first, int n) {
    TrRange nvtx("sppm.iterations");
    if (n <= 0) return 0;
    SppmState* s = c->sppm;
    struct Flag { bool& f; explicit Flag(bool& f_) : f(f_) { f = true; } ~Flag() { f = false; } } pipelined(s->pipelined);
    // Everything is enqueued on the context's high-priority chain stream, forked from / joined into the caller's stream
    // (so the caller's stream still orders everything): while this scope lives, c->stream IS the chain stream.
    struct ChainScope {
        trace_ctx* c; cudaStream_t caller; bool on;
        explicit ChainScope(trace_ctx* c_) : c(c_), caller(c_->stream), on(c_->sppm_chain_priority && c_->chain_stream) {
            if (!on) return;
            cudaEventRecord(c->ev_chain, caller);
            cudaStreamWaitEvent(c->chain_stream, c->ev_chain, 0);
            c->stream = c->cur_stream = c->chain_stream;
        }
        ~ChainScope() {
            if (!on) return;
            cudaEventRecord(c->ev_chain, c->chain_stream);
            cudaStreamWaitEvent(caller, c->ev_chain, 0);
            c->stream = c->cur_stream = caller;
        }
    } chain(c);
    const bool multi = c->comm != nullptr && c->world > 1;
    if (multi) {                                                 // the collective stream starts behind whatever the caller enqueued
        TR_CUDA(c, cudaEventRecord(c->ev_fork, c->stream));
        TR_CUDA(c, cudaStreamWaitEvent(c->coll_stream, c->ev_fork, 0));
    }
    const bool look_ahead = s->D >= 2;
    const int last = first + n - 1;
    if (sppm_phase_a(c, first)) return 1;
    for (int it = first; it <= last; ++it) {
        if (look_ahead && it < last && sppm_phase_a(c, it + 1)) return 1;
        if (sppm_phase_b(c, it)) return 1;
        if (!look_ahead && it < last && sppm_phase_a(c, it + 1)) return 1;
    }
    if (multi) {                                                 // ... and the caller's stream ends behind the collective stream
        TR_CUDA(c, cudaEventRecord(c->ev_fork, c->coll_stream));
        TR_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_fork, 0));
    }
    return 0;
}

extern "C" int trace_render_sppm(trace_ctx* c, const trace_camera* cam, const trace_film_desc* film, float r0, int max_depth,
                                 int n_iterations, int64_t photons, int write_frequency, uint64_t seed, trace_sppm_cb on_image,
                                 void* user, float* rgb_out) {
    if (!c) return 1;
    if (n_iterations < 1) return c->fail("trace_render_sppm: n_iterations must be >= 1");
    if (!rgb_out) return c->fail("trace_render_sppm: null output");
    if (c->world != 1 && !c->comm)
        return c->fail("trace_render_sppm over several ranks needs trace_comm_init (or drive the stepwise trace_sppm_* API and do the exchanges yourself)");
    if (trace_sppm_begin(c, cam, film, r0, max_depth, photons, seed)) return 1;
    TR_CUDA(c, cudaEventRecord(c->ev0, c->stream));
    // iterations are enqueued in runs that end where the caller wants an image (sppm.jl:167-171)
    const bool stream_images = on_image && write_frequency > 0;
    for (int it = 1; it <= n_iterations;) {
        int run = n_iterations - it + 1;
        if (stream_images) run = std::min(run, write_frequency - (it - 1) % write_frequency);
        if (sppm_iterations_async(c, it, run)) { sppm_end_session(c); return 1; }
        it += run;
        const int done = it - 1;
        if (stream_images && done % write_frequency == 0 && done != n_iterations) {
            if (trace_sppm_image(c, done, rgb_out)) { sppm_end_session(c); return 1; }
            on_image(user, done, rgb_out);
        }
    }
    TR_CUDA(c, cudaEventRecord(c->ev1, c->stream));
    if (trace_sppm_image(c, n_iterations, rgb_out)) { sppm_end_session(c); return 1; }      // (the one host wait; checks the error flags)
    float ms = 0.0f;
    cudaEventElapsedTime(&ms, c->ev0, c->ev1);
    c->stats.ms_total = ms;
    if (on_image) on_image(user, n_iterations, rgb_out);
    return trace_sppm_end(c);
}

// Session form of the same loop for callers that keep iterating (animations, benchmarks): trace_sppm_begin, then
// trace_sppm_iterate(n) as often as wanted - n iterations are enqueued back to back, no host wait - then trace_sppm_image
// / trace_sppm_end.  Collectives as in trace_render_sppm when a communicator exists.
extern "C" int trace_sppm_iterate(trace_ctx* c, int first_iteration, int n) {
    if (!c) return 1;
    cudaSetDevice(c->device);
    if (!c->sppm || !c->sppm->active) return c->fail("trace_sppm_iterate: call trace_sppm_begin first");
    if (first_iteration < 1 || n < 0) return c->fail("trace_sppm_iterate: bad arguments");
    if (c->world != 1 && !c->comm) return c->fail("trace_sppm_iterate over several ranks needs trace_comm_init");
    return sppm_iterations_async(c, first_iteration, n);
}
