// whitted.cu — wavefront Whitted integrator: generate -> extend (closest hit) -> shade -> shadow (any hit) ->
// accumulate, with SoA float4 ray / hit / shadow queues in HBM and warp-aggregated atomic compaction between stages.
//
// Replaces (i::SamplerIntegrator)(scene), li, specular_reflect, specular_transmit (src/integrators/sampler.jl:12-199)
// and add_sample! / merge_film_tile! (src/film.jl:134-193).
//
// The reference's `li` is a depth-first recursion that returns L bottom-up; here every ray carries the product of
// the f·|cos|/pdf factors above it (its weight), every shadow ray carries weight·f·Li·|cos|/pdf, and an unoccluded
// shadow ray adds that to the per-sample accumulator.  A sample is splatted into the film only when its whole ray
// tree has drained, which keeps the reference's per-sample `isnan(l) -> 0` rule (sampler.jl:46).
//
// Slot layout of one batch: slot = (local tile, pixel in tile, sample); 32 consecutive slots are 2 pixels x 16 spp or
// (spp = 1) two 16-pixel rows of one 16x16 tile, so primary rays of a warp are coherent.
#include "context.hpp"
#include "shading.cuh"
#include "wavefront.cuh"

// what may change between two renders that replay the same CUDA graph: read through a pointer, not baked into a node
struct WhittedFrame {
    DeviceCamera cam;
    uint64_t seed;
};

struct WhittedLaunch {
    DeviceScene sc;
    const WhittedFrame* frame;
    DeviceFilm film;
    int spp, max_depth;
    long long slot_begin;      // first slot of this batch (global over the rank's tile list); a multiple of 256 * spp
    int n_slots;
    int tile_begin;            // slot_begin / (256 * spp): first entry of `tiles` this batch covers
    int spp_shift;             // log2(spp) when spp is a power of two, else -1
    int fused;                 // 1: no primary-ray queue - k_wh_primary generates and traces, shade / splat re-derive the ray
    const int* tiles;          // tile indices owned by this rank
    float4 *ro[2], *rd[2], *rw[2];   // ray queues: {o, tmax} {d, slot} {weight, -}
    float4* hits;              // {b2, prim+1 (bits), b0, b1}
    float4 *so, *sd, *sc_contrib;     // shadow queue: {o,-} {d, slot} {contribution,-}
    float4* accum;             // per slot: radiance
    float2* filmpos;           // per slot: p_film (x < -1e29: inactive slot)
    int* counters;             // [level] rays in queue at that level (1-based), [32] shadow rays of the whole batch
    int cap_rays, cap_shadow;
    float4* film_rgbw;         // per film pixel: sum(L*w) rgb, sum(w)
    unsigned long long* stats; // u64 statistics block of the context
};

// slot (batch-local, 32-bit) -> pixel, sample, tile.  Batches start on tile boundaries, so no 64-bit arithmetic; with a
// power-of-two spp (every config) the two divisions are shifts.
__device__ __forceinline__ void slot_to_pixel(const WhittedLaunch& L, int i, int& px, int& py, int& s, int& tile) {
    unsigned lt, pix;
    const unsigned u = (unsigned)i;
    if (L.spp_shift >= 0) {
        lt = u >> (8 + L.spp_shift);
        const unsigned within = u & ((256u << L.spp_shift) - 1u);
        pix = within >> L.spp_shift;
        s = (int)(within & ((1u << L.spp_shift) - 1u));
    } else {
        const unsigned per_tile = 256u * (unsigned)L.spp;
        lt = u / per_tile;
        const unsigned within = u - lt * per_tile;
        pix = within / (unsigned)L.spp;
        s = (int)(within - pix * (unsigned)L.spp);
    }
    tile = __ldg(&L.tiles[L.tile_begin + (int)lt]);
    const int ty = tile / L.film.tiles_x, tx = tile - ty * L.film.tiles_x;
    px = L.film.sb_x0 + tx * 16 + (int)(pix & 15u);
    py = L.film.sb_y0 + ty * 16 + (int)(pix >> 4);
}

// the camera sample of a slot: film position (px + u0, py + u1) and its ray.  Pure function of (seed, pixel, sample),
// so the fused path re-derives it in shade and splat instead of storing it.  Returns false for slots outside the
// sample bounds (tiles overhang the image).
__device__ __forceinline__ bool slot_film_position(const WhittedLaunch& L, uint64_t seed, int i, int& px, int& py, int& s, int& tile,
                                                   uint32_t& pix, float& fx, float& fy) {
    slot_to_pixel(L, i, px, py, s, tile);
    if (px > L.film.sb_x1 || py > L.film.sb_y1) return false;
    pix = (uint32_t)((py - L.film.sb_y0) * (L.film.sb_x1 - L.film.sb_x0 + 1) + (px - L.film.sb_x0));
    fx = (float)px + rng_uniform(seed, pix, (uint32_t)s, 0);
    fy = (float)py + rng_uniform(seed, pix, (uint32_t)s, 1);
    return true;
}
__device__ __forceinline__ void slot_camera_ray(const DeviceCamera& cam, uint64_t seed, uint32_t pix, int s, float fx, float fy,
                                                float3& o, float3& d) {
    float l0 = 0.0f, l1 = 0.0f;
    if (cam.lens_radius > 0.0f) { l0 = rng_uniform(seed, pix, (uint32_t)s, 2); l1 = rng_uniform(seed, pix, (uint32_t)s, 3); }
    generate_camera_ray(cam, fx, fy, l0, l1, o, d);
}

// unfused path (instrumented passes): one camera ray per slot into the level-1 queue
__global__ void __launch_bounds__(256) k_wh_generate(WhittedLaunch L) {
    const DeviceCamera cam = L.frame->cam;
    const uint64_t seed = L.frame->seed;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < L.n_slots; i += gridDim.x * blockDim.x) {
        int px, py, s, tile;
        uint32_t pix;
        float fx, fy;
        L.accum[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (!slot_film_position(L, seed, i, px, py, s, tile, pix, fx, fy)) { L.filmpos[i] = make_float2(-1e30f, -1e30f); continue; }
        L.filmpos[i] = make_float2(fx, fy);
        float3 o, d;
        slot_camera_ray(cam, seed, pix, s, fx, fy, o, d);
        const int q = queue_claim(&L.counters[1]);
        L.ro[0][q] = f4(o, TR_INF);
        L.rd[0][q] = f4(d, __int_as_float(i));
        L.rw[0][q] = make_float4(1.0f, 1.0f, 1.0f, 0.0f);
    }
}

// fused path: generate the camera ray of slot i and trace it right away - hit record i belongs to slot i, there is no
// primary-ray queue (saves writing and re-reading 48 bytes per sample and one launch per batch)
// the camera sample of slot i as a call (not inlined): its ~40 live values stay out of the traversal loop's registers
static __device__ __noinline__ bool primary_ray(const WhittedLaunch& L, int i, float3& o, float3& d) {
    int px, py, s, tile;
    uint32_t pix = 0;
    float fx, fy;
    const uint64_t seed = L.frame->seed;
    if (!slot_film_position(L, seed, i, px, py, s, tile, pix, fx, fy)) return false;
    slot_camera_ray(L.frame->cam, seed, pix, s, fx, fy, o, d);
    return true;
}

// TREE: walk the shadow tree (traverse_closest); L.sc is then the launch's hit_launch_scene
template <int SLAB, int WAIT, bool TREE>
__global__ void __launch_bounds__(128, TR_TRAV_MIN_BLOCKS) k_wh_primary(const __grid_constant__ WhittedLaunch L, int* error_flag) {
    const int lane = threadIdx.x & 31;
    int n_active = 0;
    for (int base = blockIdx.x * blockDim.x + (threadIdx.x - lane); base < L.n_slots; base += gridDim.x * blockDim.x) {
        const int i = base + lane;
        float3 o = f3s(0.0f), d = f3s(1.0f);
        const bool valid = i < L.n_slots && primary_ray(L, i, o, d);
        // the ray generation above diverges (sample bounds, w == 1 shortcut of the projective divide, lens) and the
        // compiler does not reconverge the warp before the traversal loop by itself: ncu showed 7 of 32 lanes per
        // instruction and 3x the run time without this barrier
        __syncwarp();
        HitRecord h;
        // counters: only the shadow-tree walk's fallback count (COUNT is off)
        traverse_closest<SLAB, false, WAIT, TREE>(L.sc, valid, o, d, TR_INF, h, L.stats + ST_NODES, error_flag);
        if (i < L.n_slots) {
            L.accum[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            q_store(&L.hits[i], make_float4(h.t, __uint_as_float(valid ? h.prim : 0u), h.b0, h.b1));
        }
        n_active += __popc(__ballot_sync(0xffffffffu, valid));
    }
    if (lane == 0 && n_active) atomicAdd(&L.counters[1], n_active);     // rays traced at level 1 (statistics only)
}

#ifndef TR_SHADE_MIN_BLOCKS
#define TR_SHADE_MIN_BLOCKS 8      // 64 registers: the shade kernels wait on scattered primitive / normal fetches, occupancy beats registers (22.75 -> 22.57 ms)
#endif
__global__ void __launch_bounds__(128, TR_SHADE_MIN_BLOCKS) k_wh_shade(WhittedLaunch L, int level) {
    const int cur = (level - 1) & 1, nxt = level & 1;
    const bool rederive = L.fused && level == 1;
    // levels >= 2 read a two-ended queue (wavefront.cuh): reflected rays from the front, transmitted rays from the back
    int nf, n;
    queue_extent(&L.counters[level], level >= 2 ? &L.counters[IC_BACK + level] : nullptr, L.cap_rays, nf, n);
    if (rederive) nf = n = L.n_slots;
    if (level >= 2 && (long long)L.counters[level] + (long long)L.counters[IC_BACK + level] > (long long)L.cap_rays)
        L.counters[IC_OVERFLOW] = 1;                           // the two ends met: the batch is re-run in halves
    if (level == 1 && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&L.stats[ST_PRIMARY_RAYS], (unsigned long long)L.counters[1]);
    unsigned n_hit = 0;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
        const int i = queue_position(j, nf, L.cap_rays);
        const float4 h = q_load(&L.hits[i]);                // queues are streamed once: keep them out of the way of the BVH in L2
        const uint32_t prim1 = __float_as_uint(h.y);
        if (prim1 == 0u) continue;                          // miss: le(light, ray) == 0 (lights/light.jl:41)
        n_hit++;
        float4 o4, d4;
        float3 w;
        if (rederive) {
            int px, py, s, tile;
            uint32_t pix;
            float fx, fy;
            slot_film_position(L, L.frame->seed, i, px, py, s, tile, pix, fx, fy);
            float3 o, dd;
            slot_camera_ray(L.frame->cam, L.frame->seed, pix, s, fx, fy, o, dd);
            o4 = f4(o, TR_INF); d4 = f4(dd, __int_as_float(i)); w = f3s(1.0f);
        } else { o4 = q_load(&L.ro[cur][i]); d4 = q_load(&L.rd[cur][i]); w = xyz(q_load(&L.rw[cur][i])); }
        float3 d = xyz(d4);
        if (d.x == 0.0f) d.x = 0.0f;                        // the ray as intersect! left it (check_direction!)
        if (d.y == 0.0f) d.y = 0.0f;
        if (d.z == 0.0f) d.z = 0.0f;
        const uint32_t prim = prim1 - 1u;
        const float b2 = third_barycentric(L.sc, prim, xyz(o4), d);
        const Interaction it = build_interaction(L.sc, prim, xyz(o4), d, h.z, h.w, b2);
        const Frame fr = make_frame(it);
        LobeSet lobes;
        material_lobes(L.sc.materials[it.material], false, lobes);
        // direct lighting: one shadow ray per light (sampler.jl:83-92)
        for (int li = 0; li < L.sc.n_lights; ++li) {
            float3 wi, lpos;
            const float3 Li = sample_li_any(L.sc.lights[li], it.p, wi, lpos);
            if (is_black3(Li)) continue;
            const float3 f = bsdf_f(lobes, fr, it.wo, wi, LB_ALL);
            if (is_black3(f)) continue;
            const float3 contrib = w * ((f * Li) * fabsf(dot3(wi, it.ns)) / 1.0f);
            const float3 sdir = lpos - it.p;                 // spawn_ray(p0, p1): un-normalised, t_max = Inf (Q5)
            const int q = queue_claim(&L.counters[32]);
            if (q < L.cap_shadow) {
                q_store(&L.so[q], f4(it.p + 1e-6f * sdir, TR_INF));
                q_store(&L.sd[q], f4(sdir, d4.w));
                q_store(&L.sc_contrib[q], f4(contrib, 0.0f));
            } else L.counters[IC_OVERFLOW] = 1;
        }
        if (level + 1 <= L.max_depth) {
            // specular_reflect / specular_transmit (sampler.jl:103-199); u is irrelevant for the delta lobes
            #pragma unroll
            for (int pass = 0; pass < 2; ++pass) {
                const uint32_t type = (pass == 0 ? LB_REFLECTION : LB_TRANSMISSION) | LB_SPECULAR;
                const BSDFSample bs = bsdf_sample(lobes, fr, it.wo, 0.5f, 0.5f, type);
                const float adot = fabsf(dot3(bs.wi, it.ns));
                if (!(bs.pdf > 0.0f && !is_black3(bs.f) && adot != 0.0f)) continue;
                const float3 wn = w * (bs.f * adot / bs.pdf);
                // reflected rays fill the next level's queue from the front, transmitted rays from the back
                const int k = queue_claim(&L.counters[(pass == 0 ? 0 : IC_BACK) + level + 1]);
                const int q = pass == 0 ? k : L.cap_rays - 1 - k;
                if (k < L.cap_rays) {
                    q_store(&L.ro[nxt][q], f4(it.p + 1e-6f * bs.wi, TR_INF));     // spawn_ray(si, wi), Trace.jl:206-211
                    q_store(&L.rd[nxt][q], f4(bs.wi, d4.w));
                    q_store(&L.rw[nxt][q], f4(wn, 0.0f));
                } else L.counters[IC_OVERFLOW] = 1;
            }
        }
    }
    if (level == 1) {                                        // primary hit fraction (reported by bench.py)
        __syncwarp();
        n_hit = __reduce_add_sync(0xffffffffu, n_hit);
        if ((threadIdx.x & 31) == 0 && n_hit) atomicAdd(&L.stats[ST_PRIMARY_HITS], (unsigned long long)n_hit);
    }
}

// add_sample! with the reference's footprint / table indexing quirks (film.jl:134-164, Q4) and the clipping to the
// FilmTile bounds of the sample's 16x16 tile (film.jl:120-125).
struct SplatClip { float x0, y0, x1, y1; };      // pixels a sample of this tile may touch (tile bounds ^ crop window)
__device__ __forceinline__ SplatClip splat_clip(const DeviceFilm& F, int tile) {
    const int ty = tile / F.tiles_x, tx = tile - ty * F.tiles_x;
    const int bx0 = F.sb_x0 + tx * 16, by0 = F.sb_y0 + ty * 16;
    const int bx1 = min(bx0 + 15, F.sb_x1), by1 = min(by0 + 15, F.sb_y1);
    SplatClip c;
    c.x0 = fmaxf(fmaxf(ceilf((float)bx0 - 0.5f - F.rx), (float)F.crop_x0), 1.0f);
    c.y0 = fmaxf(fmaxf(ceilf((float)by0 - 0.5f - F.ry), (float)F.crop_y0), 1.0f);
    c.x1 = fminf(floorf((float)bx1 - 0.5f + F.rx) + 1.0f, (float)F.crop_x1);
    c.y1 = fminf(floorf((float)by1 - 0.5f + F.ry) + 1.0f, (float)F.crop_y1);
    return c;
}
// does sample (dx, dy) touch pixel (x, y), and with which filter weight
__device__ __forceinline__ bool splat_weight(const DeviceFilm& F, const SplatClip& c, float dx, float dy, float x, float y, float& wgt) {
    const float p0x = fmaxf(ceilf(dx - F.rx), c.x0), p0y = fmaxf(ceilf(dy - F.ry), c.y0);
    const float p1x = fminf(floorf(dx + F.rx) + 1.0f, c.x1), p1y = fminf(floorf(dy + F.ry) + 1.0f, c.y1);
    if (x < p0x || x > p1x || y < p0y || y > p1y) return false;
    const int oy = (int)clampf(floorf(fabsf((y - dy) * F.inv_ry * 16.0f)), 1.0f, 16.0f);
    const int ox = (int)clampf(ceilf(fabsf((x - dx) * F.inv_rx * 16.0f)), 1.0f, 16.0f);
    wgt = __ldg(&F.table[(oy - 1) * 16 + (ox - 1)]);
    return true;
}

// One film atomic per (pixel, touched film pixel) instead of one per (sample, touched film pixel): with spp a multiple
// of 16 the 16 lanes of a half-warp hold 16 samples of ONE pixel; their footprints lie in a small common window
// ((2r + 3)^2 film pixels: 4 x 4 for the radius-1 filter of every config), so each lane takes one film pixel of the
// window, gathers the 16 samples by shuffle and issues one 128-bit atomic (round 1: 9 atomics per sample, the kernel
// was bound by L2 atomic throughput).  Other spp values use the per-sample path.
__global__ void __launch_bounds__(256) k_wh_splat(WhittedLaunch L) {
    if (L.counters[IC_OVERFLOW]) return;                      // the host re-runs the batch in smaller pieces
    const DeviceFilm& F = L.film;
    const uint64_t seed = L.frame->seed;
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const bool grouped = (L.spp & 15) == 0;
    for (int base = blockIdx.x * blockDim.x + (threadIdx.x - lane); base < L.n_slots; base += gridDim.x * blockDim.x) {
        const int i = base + lane;
        int px = 0, py = 0, s, tile = 0;
        uint32_t pix;
        float fx = 0.0f, fy = 0.0f;
        bool valid = i < L.n_slots;
        if (valid) {
            if (L.fused) valid = slot_film_position(L, seed, i, px, py, s, tile, pix, fx, fy);
            else {
                const float2 fp = L.filmpos[i];
                valid = !(fp.x < -1e29f);
                fx = fp.x; fy = fp.y;
                slot_to_pixel(L, i, px, py, s, tile);
            }
        }
        float4 a = valid ? L.accum[i] : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (isnan(a.x) || isnan(a.y) || isnan(a.z)) { a.x = 0.0f; a.y = 0.0f; a.z = 0.0f; }      // sampler.jl:46
        const float dx = fx - 0.5f, dy = fy - 0.5f;
        if (!grouped) {
            if (!valid) continue;
            const SplatClip c = splat_clip(F, tile);
            const float p0x = fmaxf(ceilf(dx - F.rx), c.x0), p0y = fmaxf(ceilf(dy - F.ry), c.y0);
            const float p1x = fminf(floorf(dx + F.rx) + 1.0f, c.x1), p1y = fminf(floorf(dy + F.ry) + 1.0f, c.y1);
            for (float y = p0y; y <= p1y; y += 1.0f)
                for (float x = p0x; x <= p1x; x += 1.0f) {
                    float wgt = 0.0f;
                    splat_weight(F, c, dx, dy, x, y, wgt);
                    const int ix = (int)x - F.crop_x0, iy = (int)y - F.crop_y0;
                    atomicAdd(&L.film_rgbw[(size_t)iy * F.width + ix], make_float4(a.x * wgt, a.y * wgt, a.z * wgt, wgt));
                }
            continue;
        }
        // grouped: the half-warp's pixel (identical in its 16 lanes) and the window its samples can touch
        const int g = lane & 15, gbase = lane & 16;
        const SplatClip c = splat_clip(F, tile);
        const float wx0 = ceilf((float)px - 0.5f - F.rx), wy0 = ceilf((float)py - 0.5f - F.ry);
        const int wnx = (int)(floorf((float)px + 0.5f + F.rx) + 1.0f - wx0) + 1, wny = (int)(floorf((float)py + 0.5f + F.ry) + 1.0f - wy0) + 1;
        const int n_targets = __shfl_sync(full, valid ? wnx * wny : 0, gbase);
        const int n_loop = max(__shfl_sync(full, n_targets, 0), __shfl_sync(full, n_targets, 16));     // warp-uniform trip count
        const bool packed = __all_sync(full, wnx <= 6 && wny <= 6);
        if (packed) {
            // Every lane works out ONCE, for its own sample, which filter-table column / row each window column / row
            // gets (0: outside the sample's footprint) - 5 bits each - so a target lane needs two shuffles and a table
            // lookup per sample instead of redoing the footprint arithmetic 16 x 16 times per pixel.
            const float p0x = fmaxf(ceilf(dx - F.rx), c.x0), p0y = fmaxf(ceilf(dy - F.ry), c.y0);
            const float p1x = fminf(floorf(dx + F.rx) + 1.0f, c.x1), p1y = fminf(floorf(dy + F.ry) + 1.0f, c.y1);
            unsigned colbits = 0u, rowbits = 0u;
            #pragma unroll
            for (int k = 0; k < 6; ++k) {
                const float x = wx0 + (float)k, y = wy0 + (float)k;
                if (valid && k < wnx && x >= p0x && x <= p1x)
                    colbits |= (unsigned)(int)clampf(ceilf(fabsf((x - dx) * F.inv_rx * 16.0f)), 1.0f, 16.0f) << (5 * k);
                if (valid && k < wny && y >= p0y && y <= p1y)
                    rowbits |= (unsigned)(int)clampf(floorf(fabsf((y - dy) * F.inv_ry * 16.0f)), 1.0f, 16.0f) << (5 * k);
            }
            for (int j0 = 0; j0 < n_loop; j0 += 16) {
                const int j = j0 + g;
                const int tyi = j / wnx, txi = j - tyi * wnx;
                float4 acc = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                bool any = false;
                #pragma unroll 4
                for (int k = 0; k < 16; ++k) {
                    const int src = gbase + k;
                    const unsigned cb = __shfl_sync(full, colbits, src), rb = __shfl_sync(full, rowbits, src);
                    const float ar = __shfl_sync(full, a.x, src), ag = __shfl_sync(full, a.y, src), ab = __shfl_sync(full, a.z, src);
                    const unsigned ox = (cb >> (5 * txi)) & 31u, oy = (rb >> (5 * tyi)) & 31u;
                    if (j < n_targets && ox != 0u && oy != 0u) {
                        const float wgt = __ldg(&F.table[(oy - 1u) * 16u + (ox - 1u)]);
                        acc.x += ar * wgt; acc.y += ag * wgt; acc.z += ab * wgt; acc.w += wgt; any = true;
                    }
                }
                if (any) {
                    const int ix = (int)wx0 + txi - F.crop_x0, iy = (int)wy0 + tyi - F.crop_y0;
                    atomicAdd(&L.film_rgbw[(size_t)iy * F.width + ix], acc);
                }
            }
            continue;
        }
        for (int j0 = 0; j0 < n_loop; j0 += 16) {          // wide filters: per-(sample, target) footprint arithmetic
            const int j = j0 + g;
            const float x = wx0 + (float)(j % wnx), y = wy0 + (float)(j / wnx);
            float4 acc = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            bool any = false;
            #pragma unroll 4
            for (int k = 0; k < 16; ++k) {
                const int src = gbase + k;
                const float kx = __shfl_sync(full, dx, src), ky = __shfl_sync(full, dy, src);
                const float ar = __shfl_sync(full, a.x, src), ag = __shfl_sync(full, a.y, src), ab = __shfl_sync(full, a.z, src);
                float wgt;
                if (j < n_targets && splat_weight(F, c, kx, ky, x, y, wgt)) {
                    acc.x += ar * wgt; acc.y += ag * wgt; acc.z += ab * wgt; acc.w += wgt; any = true;
                }
            }
            if (any) {
                const int ix = (int)x - F.crop_x0, iy = (int)y - F.crop_y0;
                atomicAdd(&L.film_rgbw[(size_t)iy * F.width + ix], acc);
            }
        }
    }
}

// merge into the caller's film: xyz += to_XYZ(contrib), weight += w (film.jl:182-193)
// `skip` (device flag, may be null): set when a batch of this render overflowed a queue or a traversal failed - the host
// then repairs the render and finalizes again, unconditionally.
__global__ void k_film_finalize(const float4* __restrict__ rgbw, float4* __restrict__ film, int n, const int* __restrict__ skip) {
    if (skip && *skip) return;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 c = rgbw[i];
        float4 f = film[i];
        f.x += (0.412453f * c.x + 0.357580f * c.y) + 0.180423f * c.z;
        f.y += (0.212671f * c.x + 0.715160f * c.y) + 0.072169f * c.z;
        f.z += (0.019334f * c.x + 0.119193f * c.y) + 0.950227f * c.z;
        f.w += c.w;
        film[i] = f;
    }
}

// Film sum + merge over peer memory: ONE kernel instead of an NCCL collective followed by the merge.  peers.film[r] is
// rank r's private film (mapped into this process, comm.cpp); this rank owns pixels [p0, p0 + n): it reads them from all
// `world` films over NVLink (ld.cv: never from a stale L1 line), sums them in rank order (deterministic, unlike a ring) and
// either merges the sum into the caller's film (film_mode 1: XYZ conversion + add, as k_film_finalize) or stores it into
// rank 0's "summed film" region (film_mode 0: rank 0 merges the whole film after the closing barrier).
struct FilmPeers { const float4* film[8]; float4* summed_on_root; };
__global__ void __launch_bounds__(256) k_film_sum_p2p(FilmPeers peers, int world, long long p0, int n, float4* __restrict__ film /* caller's, or null */,
                                                      const int* __restrict__ skip) {
    if (skip && *skip) return;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const long long px = p0 + i;
        float4 c = __ldcv(&peers.film[0][px]);
        for (int r = 1; r < world; ++r) {
            const float4 v = __ldcv(&peers.film[r][px]);
            c.x += v.x; c.y += v.y; c.z += v.z; c.w += v.w;
        }
        if (film) {
            float4 f = film[px];
            f.x += (0.412453f * c.x + 0.357580f * c.y) + 0.180423f * c.z;
            f.y += (0.212671f * c.x + 0.715160f * c.y) + 0.072169f * c.z;
            f.z += (0.019334f * c.x + 0.119193f * c.y) + 0.950227f * c.z;
            f.w += c.w;
            film[px] = f;
        } else peers.summed_on_root[px] = c;
    }
}

// any[0] = 1 when one of the render's batches overflowed or a traversal ran out of stack, any[1] = 1 for the latter alone
// (with a communicator the pair is summed over the ranks, so that all of them take the same path afterwards)
__global__ void k_wh_any_flag(const int* __restrict__ batch_flags, int n, const int* __restrict__ error_flag, int* __restrict__ any) {
    int bad = 0;
    for (int i = threadIdx.x; i < n; i += 32) bad |= batch_flags[i];
    bad = __any_sync(0xffffffffu, bad != 0);
    if (threadIdx.x == 0) { any[0] = (bad || *error_flag) ? 1 : 0; any[1] = *error_flag ? 1 : 0; }
}

__global__ void k_wh_batch_stats(int* counters, unsigned long long* stats, int max_depth, int cap_rays, int cap_shadow,
                                 int* batch_flag) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        if (batch_flag) *batch_flag = counters[IC_OVERFLOW];
        unsigned long long e = 0, s = 0;
        for (int l = 1; l <= max_depth; ++l) e += min(counters[l] + (l >= 2 ? counters[IC_BACK + l] : 0), cap_rays);
        s = min(counters[32], cap_shadow);
        if (!counters[IC_OVERFLOW]) { atomicAdd(&stats[ST_RAYS_EXTEND], e); atomicAdd(&stats[ST_RAYS_SHADOW], s); }
    }
}

// Enqueues one batch.  batch_flag == nullptr: synchronous (waits, checks the overflow flag, re-runs in halves).
// batch_flag != nullptr: asynchronous - the batch's overflow flag is left in *batch_flag (device memory) and the caller
// inspects all flags once after the last batch, so the host never waits on the GPU between batches (the per-batch
// sync cost ~0.9 ms of GPU idle time per batch on B200: 17 launches to enqueue behind an empty stream).
static int run_batch(trace_ctx* c, WhittedLaunch& L, long long begin, long long count, int depth_guard, int* batch_flag = nullptr) {
    if (count <= 0) return 0;
    TrRange nvtx_batch("whitted.batch: primary -> (extend -> shade) x depth -> shadow -> splat");
    const long long per_tile = 256ll * L.spp;
    L.slot_begin = begin;
    L.n_slots = (int)count;
    L.tile_begin = (int)(begin / per_tile);                    // batches start on tile boundaries
    // fused primary stage unless an instrumented pass needs the plain kernels (node counting)
    L.fused = (c->fuse_primary && !c->count_nodes && c->slab != 1) ? 1 : 0;
    int* ic = ctx_icounters(c);
    unsigned long long* st = ctx_stats64(c);
    TR_CUDA(c, cudaMemsetAsync(ic, 0, 60 * sizeof(int), c->cur_stream));
    TR_CUDA(c, cudaMemsetAsync(ic + 64, 0, 64 * sizeof(int), c->cur_stream)); c->work_slot = 0;
    TR_CUDA(c, cudaMemsetAsync(ic + IC_OVERFLOW, 0, sizeof(int), c->cur_stream));
    const int g_stream = persistent_grid(c, 8), g_trav = persistent_grid(c, 16);
    int* d_err = ctx_icounters_lane(c, 0) + IC_ERROR;
    if (L.fused) {
        c->kev_begin(0);
        WhittedLaunch P = L;
        P.sc = hit_launch_scene(c, L.sc);
        trav_dispatch(c, [&](auto S, auto C_, auto W) {
            constexpr int s = decltype(S)::value, w = decltype(W)::value;
            auto k = k_wh_primary<s, w, false>;
            if constexpr (shadow_walk_capable<s, false, w>) if (P.sc.shadow_pairs) k = k_wh_primary<s, w, true>;
            k<<<g_trav, 128, 0, c->cur_stream>>>(P, d_err);
        });
        c->kev_end();
    } else { c->kev_begin(TRACE_K_GENERATE); k_wh_generate<<<g_stream, 256, 0, c->cur_stream>>>(L); c->kev_end(); }
    c->stats.kernel_launches++;
    for (int level = 1; level <= L.max_depth; ++level) {
        const int cur = (level - 1) & 1;
        c->cur_level = level;
        if (!(L.fused && level == 1))
            launch_extend(c, g_trav, L.sc, (const float4*)L.ro[cur], (const float4*)L.rd[cur], (const int*)(ic + level), L.cap_rays,
                          L.hits, st + ST_NODES, d_err, level >= 2 ? (const int*)(ic + IC_BACK + level) : nullptr);
        c->kev_begin(TRACE_K_SHADE);
        k_wh_shade<<<occupancy_grid(c, k_wh_shade, 128), 128, 0, c->cur_stream>>>(L, level);
        c->kev_end();
        c->stats.kernel_launches++;
    }
    // one any-hit launch over the shadow rays of ALL bounce levels of the batch (they only feed the accumulators): a
    // single wide launch instead of max_depth launches that each wait for their slowest ray
    launch_shadow(c, g_trav, L.sc, (const float4*)L.so, (const float4*)L.sd, (const float4*)L.sc_contrib,
                  (const int*)(ic + 32), L.cap_shadow, L.accum, st + ST_NODES, d_err);
    c->kev_begin(TRACE_K_SPLAT);
    k_wh_splat<<<g_stream, 256, 0, c->cur_stream>>>(L);
    c->kev_end();
    k_wh_batch_stats<<<1, 32, 0, c->cur_stream>>>(ic, st, L.max_depth, L.cap_rays, L.cap_shadow, batch_flag);
    c->stats.kernel_launches += 2;
    TR_CUDA(c, cudaGetLastError());
    if (batch_flag) return 0;
    TR_CUDA(c, cudaMemcpyAsync(c->h_flags, ic + IC_OVERFLOW, sizeof(int), cudaMemcpyDeviceToHost, c->cur_stream));
    TR_CUDA(c, cudaMemcpyAsync(c->h_flags + 1, ctx_icounters_lane(c, 0) + IC_ERROR, sizeof(int), cudaMemcpyDeviceToHost, c->cur_stream));
    TR_CUDA(c, cudaStreamSynchronize(c->cur_stream));
    c->kev_collect();
    if (c->h_flags[1]) {
        cudaMemsetAsync(ctx_icounters_lane(c, 0) + IC_ERROR, 0, sizeof(int), c->cur_stream);
        return c->fail("traversal stack overflow (more than 64 pending nodes; the reference would throw a BoundsError, bvh.jl:222)");
    }
    if (c->h_flags[0]) {                                  // a queue overflowed: nothing was splatted, redo in halves
        c->stats.queue_overflows++;
        if (count < 2 * per_tile || depth_guard > 24) return c->fail("ray queue overflow that halving the batch cannot resolve");
        const long long half = count / 2 / per_tile * per_tile;
        if (run_batch(c, L, begin, half, depth_guard + 1)) return 1;
        return run_batch(c, L, begin + half, count - half, depth_guard + 1);
    }
    return 0;
}

// Film pixels [*p0, *p1) (row-major) this rank's film receives: everything on one GPU; with a communicator either the whole
// film on rank 0 and nothing elsewhere (film_mode 0) or the rank's chunk of ceil(n / world) pixels (film_mode 1).
void whitted_film_range(const trace_ctx* c, long long npix, long long* p0, long long* p1) {
    *p0 = 0; *p1 = npix;
    if (!c->comm || c->world <= 1) return;
    if (c->film_mode == 0) { if (c->rank != 0) *p1 = 0; return; }
    const long long chunk = (npix + c->world - 1) / c->world;
    *p0 = std::min(npix, (long long)c->rank * chunk);
    *p1 = std::min(npix, *p0 + chunk);
}

int whitted_render_device(trace_ctx* c, const trace_camera* cam, const trace_film_desc* film, int spp, int max_depth,
                          uint64_t seed, float* film_dev) {
    TrRange nvtx_render("trace_render_whitted");
    if (c->rank < 0 || c->rank >= c->world) return c->fail("rank %d outside world %d", c->rank, c->world);
    if (max_depth < 1 || max_depth > TR_MAX_DEPTH) return c->fail("max_depth must be in [1, %d]", TR_MAX_DEPTH);
    WhittedLaunch L;
    memset(&L, 0, sizeof(L));                                   // padding too: the struct's bytes key the graph cache
    L.sc = c->scene;
    WhittedFrame frame;
    memset(&frame, 0, sizeof(frame));
    ctx_device_camera(cam, &frame.cam);
    frame.seed = seed;
    TR_CUDA(c, c->b_misc[3].ensure(sizeof(WhittedFrame)));
    TR_CUDA(c, cudaMemcpyAsync(c->b_misc[3].p, &frame, sizeof(frame), cudaMemcpyHostToDevice, c->stream));
    L.frame = c->b_misc[3].as<WhittedFrame>();
    if (ctx_device_film(c, film, &L.film, &c->b_misc[0])) return 1;
    L.spp = spp; L.max_depth = max_depth;
    L.spp_shift = (spp & (spp - 1)) == 0 ? __builtin_ctz((unsigned)spp) : -1;
    // this rank's tiles: k = rank, rank + world, ...   (16x16 sample tiles, sampler.jl:24-31)
    const int total_tiles = L.film.tiles_x * L.film.tiles_y;
    std::vector<int> tiles;
    for (int k = c->rank; k < total_tiles; k += c->world) tiles.push_back(k);
    const long long total_slots = (long long)tiles.size() * 256 * spp;
    // batches of (at most) c->batch samples, evened out.  Deep bounce levels hold few but expensive rays (a launch
    // cannot end before its slowest ray: ~0.2 ms for a 1000-node walk), so batches are large and up to `lanes` of them
    // run concurrently on side streams, each lane with its own queues and counters.
    // c->batch bounds the samples in flight over ALL lanes (queue memory ~ 350 B per sample in flight)
    int K = 1;
    if (total_slots >= (long long)c->lanes * 131072) K = c->lanes;
    const long long per_lane = std::max<long long>(65536, c->batch / K);
    long long nb = std::max<long long>(K, (total_slots + per_lane - 1) / per_lane);
    nb = (nb + K - 1) / K * K;                                  // whole rounds of K lanes
    const long long per_tile = 256ll * spp;
    long long batch = (total_slots + nb - 1) / nb;
    batch = std::max<long long>(per_tile, (batch + per_tile - 1) / per_tile * per_tile);     // whole tiles: 32-bit slot math in the kernels
    if (batch > 0x7fffffffll / 2) return c->fail("batch too large: set option \"batch\" below 2^30 samples");
    nb = (total_slots + batch - 1) / batch;
    {
        // Batches are contiguous slot ranges, i.e. runs of the tile list.  In image order a run is a band of the image,
        // and bands differ wildly in cost (sky vs. geometry): lanes with cheap bands drain at once and the expensive
        // ones finish alone.  Deal groups of the rank's tiles (default: 2 tile rows - whole rows keep the BVH working set
        // of a batch compact) to the batches round-robin instead, so every batch samples the whole image.  Measured on
        // tess-1M: 1/8 of the frame 4.73 -> 4.53 ms, the full frame unchanged (profiles/r1_experiments.md).  The image
        // does not depend on the order: the RNG is keyed by the pixel.
        std::vector<int> dealt;
        dealt.reserve(tiles.size());
        const size_t G = c->deal > 0 ? (size_t)c->deal : std::max<size_t>(1, (size_t)(-c->deal) * L.film.tiles_x / c->world);
        const size_t groups = (tiles.size() + G - 1) / G;
        if (c->deal == 0) dealt = tiles;
        else
            for (long long j = 0; j < nb; ++j)
                for (size_t g = (size_t)j; g < groups; g += (size_t)nb)
                    for (size_t k = g * G; k < std::min(tiles.size(), (g + 1) * G); ++k) dealt.push_back(tiles[k]);
        tiles.swap(dealt);
    }
    TR_CUDA(c, c->b_misc[1].ensure((tiles.size() + 1) * sizeof(int)));
    if (c->wh_tiles_dev != c->b_misc[1].p || c->wh_tiles != tiles) {        // (re-rendering the same film: already there)
        if (!tiles.empty()) TR_CUDA(c, cudaMemcpyAsync(c->b_misc[1].p, tiles.data(), tiles.size() * sizeof(int), cudaMemcpyHostToDevice, c->stream));
        TR_CUDA(c, cudaStreamSynchronize(c->stream));
        c->wh_tiles = tiles; c->wh_tiles_dev = c->b_misc[1].p;
    }
    L.tiles = c->b_misc[1].as<int>();
    std::vector<long long> b_begin, b_count;
    for (long long bi = 0; bi < nb; ++bi) { b_begin.push_back(bi * batch); b_count.push_back(std::min(batch, total_slots - bi * batch)); }
    const size_t cap_rays = (size_t)batch * (size_t)c->cap_percent / 100;
    const int shadow_mult = std::max(1, std::min(L.sc.n_lights, 4));
    const size_t cap_shadow = cap_rays * shadow_mult * 2;     // all bounce levels of a batch share one shadow queue
    L.cap_rays = (int)cap_rays; L.cap_shadow = (int)cap_shadow;
    for (int k = 0; k < 7; ++k) TR_CUDA(c, c->b_queue[k].ensure(K * cap_rays * sizeof(float4)));
    for (int k = 7; k < 10; ++k) TR_CUDA(c, c->b_queue[k].ensure(K * cap_shadow * sizeof(float4)));
    TR_CUDA(c, c->b_queue[10].ensure((size_t)K * batch * sizeof(float4)));
    TR_CUDA(c, c->b_queue[11].ensure((size_t)K * batch * sizeof(float2)));
    const size_t npix = (size_t)L.film.width * L.film.height;
    const size_t npix_padded = (npix + (size_t)c->world - 1) / (size_t)c->world * (size_t)c->world;     // equal chunks for the reduce-scatter
    // With a communicator of <= 8 ranks the private film lives in an allocation the other ranks map (peer-memory film
    // sum, see k_film_sum_p2p): [private film | summed film].  The mappings are exchanged once per film size - a
    // collective step, taken by all ranks in the same render because they all render the same film.
    const bool want_p2p = c->comm != nullptr && c->world > 1 && c->world <= 8 && c->film_p2p;
    if (want_p2p && (c->p2p_npix != npix_padded || c->p2p_state == 0)) {
        TR_CUDA(c, cudaStreamSynchronize(c->stream));
        comm_p2p_close(c);
        c->p2p_film.release();
        TR_CUDA(c, c->p2p_film.ensure(2 * npix_padded * sizeof(float4)));
        int all_ok = 0;
        if (comm_p2p_exchange(c, c->p2p_film.p, c->p2p_peer, c->p2p_opened, &all_ok)) return 1;
        c->p2p_state = all_ok ? 1 : -1;
        c->p2p_npix = npix_padded;
        if (getenv("TRACE_CUDA_VERBOSE"))
            fprintf(stderr, "[trace_cuda rank %d] peer-memory film sum %s (%d ranks, %zu film pixels)\n", c->rank,
                    all_ok ? "enabled" : "unavailable: staying on NCCL", c->world, npix);
        c->wh_graph_key.clear();
    }
    const bool p2p = want_p2p && c->p2p_state == 1;
    if (p2p) L.film_rgbw = c->p2p_film.as<float4>();
    else {
        TR_CUDA(c, c->b_queue[12].ensure(npix_padded * sizeof(float4)));
        L.film_rgbw = c->b_queue[12].as<float4>();
    }
    L.stats = ctx_stats64(c);
    std::vector<WhittedLaunch> lane((size_t)K, L);
    for (int l = 0; l < K; ++l) {
        WhittedLaunch& W = lane[l];
        W.ro[0] = c->b_queue[0].as<float4>() + l * cap_rays; W.ro[1] = c->b_queue[1].as<float4>() + l * cap_rays;
        W.rd[0] = c->b_queue[2].as<float4>() + l * cap_rays; W.rd[1] = c->b_queue[3].as<float4>() + l * cap_rays;
        W.rw[0] = c->b_queue[4].as<float4>() + l * cap_rays; W.rw[1] = c->b_queue[5].as<float4>() + l * cap_rays;
        W.hits = c->b_queue[6].as<float4>() + l * cap_rays;
        W.so = c->b_queue[7].as<float4>() + l * cap_shadow; W.sd = c->b_queue[8].as<float4>() + l * cap_shadow;
        W.sc_contrib = c->b_queue[9].as<float4>() + l * cap_shadow;
        W.accum = c->b_queue[10].as<float4>() + (size_t)l * batch; W.filmpos = c->b_queue[11].as<float2>() + (size_t)l * batch;
        W.counters = ctx_icounters_lane(c, l);
    }
    TR_CUDA(c, c->b_misc[2].ensure((size_t)(nb + 4) * sizeof(int)));
    int* d_flags = c->b_misc[2].as<int>();
    TR_CUDA(c, cudaEventRecord(c->ev0, c->stream));
    // everything up to the lanes' join: film clear, then batch bi on lane bi % K
    auto enqueue = [&]() -> int {
        TR_CUDA(c, cudaMemsetAsync(L.film_rgbw, 0, npix_padded * sizeof(float4), c->stream));
        if (K > 1) {
            TR_CUDA(c, cudaEventRecord(c->ev_fork, c->stream));
            for (int l = 0; l < K; ++l) TR_CUDA(c, cudaStreamWaitEvent(c->side[l], c->ev_fork, 0));
        }
        int rc = 0;
        for (long long bi = 0; bi < nb && !rc; ++bi) {
            const int l = (int)(bi % K);
            c->cur_lane = l;
            c->cur_stream = K > 1 ? c->side[l] : c->stream;
            rc = run_batch(c, lane[l], b_begin[bi], b_count[bi], 0, d_flags + bi);
        }
        if (K > 1) {
            for (int l = 0; l < K; ++l) {
                cudaEventRecord(c->ev_join[l], c->side[l]);
                cudaStreamWaitEvent(c->stream, c->ev_join[l], 0);
            }
        }
        c->cur_lane = 0;
        c->cur_stream = c->stream;
        return rc;
    };
    int rc = 0;
    if (c->graph && !c->time_kernels && (size_t)c->stream > 2) {       // (legacy / per-thread default streams cannot be captured)
        std::string key((const char*)lane.data(), lane.size() * sizeof(WhittedLaunch));
        key.append((const char*)b_count.data(), b_count.size() * sizeof(long long));
        const long long extra[] = {nb, batch, K, total_slots, (long long)(size_t)d_flags, c->slab, c->persist, c->count_nodes, c->leaf_wait, c->fuse_primary, c->shadow_tree, c->hit_tree,
                                   (long long)(size_t)c->stream};
        key.append((const char*)extra, sizeof(extra));
        if (!c->wh_graph || key != c->wh_graph_key) {
            if (c->wh_graph) { cudaGraphExecDestroy(c->wh_graph); c->wh_graph = nullptr; }
            const unsigned long long before = c->stats.kernel_launches;
            TR_CUDA(c, cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeRelaxed));
            rc = enqueue();
            cudaGraph_t g = nullptr;
            const cudaError_t e_end = cudaStreamEndCapture(c->stream, &g);
            c->wh_graph_launches[0] = c->stats.kernel_launches - before;
            c->stats.kernel_launches = before;
            if (rc || e_end != cudaSuccess) {
                if (g) cudaGraphDestroy(g);
                cudaGetLastError();
                return rc ? 1 : c->fail("CUDA graph capture of the render failed: %s", cudaGetErrorString(e_end));
            }
            const cudaError_t e_inst = cudaGraphInstantiate(&c->wh_graph, g, 0);
            cudaGraphDestroy(g);
            if (e_inst != cudaSuccess) { c->wh_graph = nullptr; return c->fail("cudaGraphInstantiate: %s", cudaGetErrorString(e_inst)); }
            c->wh_graph_key = key;
        }
        TR_CUDA(c, cudaGraphLaunch(c->wh_graph, c->stream));
        c->stats.kernel_launches += c->wh_graph_launches[0];
    } else {
        rc = enqueue();
    }
    if (rc) return 1;
    int* d_err = ctx_icounters_lane(c, 0) + IC_ERROR;
    const bool multi = c->comm != nullptr && c->world > 1;
    long long f0 = 0, f1 = (long long)npix;                     // film pixels this rank delivers
    whitted_film_range(c, (long long)npix, &f0, &f1);
    // The ONE exchange of a multi-rank render (SURVEY.md 8e): the sum of the ranks' private films, on the render's stream.
    // Peer-memory form: [barrier: every rank's private film is final] -> k_film_sum_p2p (sum + merge of this rank's pixels,
    // read from all ranks' films) -> [barrier: nobody reads a private film any more, so the next render may clear it;
    // film_mode 0: all bands have landed in rank 0's summed film] -> (film_mode 0, rank 0) merge of the whole film.  The
    // barriers are one-int all-reduces; the first one is the flag all-reduce of the render when it directly precedes.
    auto film_sum_p2p = [&](bool need_open_barrier, const int* skip) -> int {
        TrRange nvtx_sum("whitted.film sum + merge (peer memory)");
        c->kev_begin(TRACE_K_COMM);
        int* d_bar = d_flags + nb + 2;
        if (need_open_barrier && comm_allreduce_sum_int(c, d_bar, 1)) return 1;
        FilmPeers peers;
        for (int r = 0; r < 8; ++r) peers.film[r] = r < c->world ? reinterpret_cast<const float4*>(c->p2p_peer[(size_t)r]) : nullptr;
        peers.summed_on_root = reinterpret_cast<float4*>(c->p2p_peer[0]) + npix_padded;
        const size_t chunk = (npix + (size_t)c->world - 1) / (size_t)c->world;
        const long long q0 = (long long)std::min(npix, (size_t)c->rank * chunk), q1 = (long long)std::min(npix, (size_t)(c->rank + 1) * chunk);
        if (q1 > q0) {
            if (c->film_mode == 1 && c->film_upload_pending) { TR_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_copy, 0)); c->film_upload_pending = false; }
            k_film_sum_p2p<<<persistent_grid(c, 4), 256, 0, c->stream>>>(peers, c->world, q0, (int)(q1 - q0),
                                                                         c->film_mode == 1 ? (float4*)film_dev : nullptr, skip);
            c->stats.kernel_launches++;
        }
        if (comm_allreduce_sum_int(c, d_bar + 1, 1)) return 1;
        c->kev_end();
        if (c->film_mode == 0 && c->rank == 0) {
            if (c->film_upload_pending) { TR_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_copy, 0)); c->film_upload_pending = false; }
            k_film_finalize<<<persistent_grid(c, 4), 256, 0, c->stream>>>(c->p2p_film.as<float4>() + npix_padded, (float4*)film_dev, (int)npix, skip);
            c->stats.kernel_launches++;
        }
        return 0;
    };
    auto film_sum = [&]() -> int {
        TrRange nvtx_sum("whitted.film sum (NCCL)");
        float* rgbw = reinterpret_cast<float*>(L.film_rgbw);
        c->kev_begin(TRACE_K_COMM);
        int rc2 = 0;
        if (c->film_mode == 0) {
            // whole film onto rank 0 (option film_sum): 0 ncclReduce, 1 ncclAllReduce, 2 (default) reduce-scatter + gather of
            // the summed chunks - measured on 8 B200: ncclReduce of the 33 MB film 0.26 ms, all-reduce no better
            if (c->film_sum == 1) rc2 = comm_allreduce_sum(c, rgbw, npix * 4);
            else if (c->film_sum == 2) rc2 = comm_reduce_sum_via_scatter(c, rgbw, (npix + (size_t)c->world - 1) / (size_t)c->world * 4, 0);
            else rc2 = comm_reduce_sum(c, rgbw, rgbw, npix * 4, 0);
        } else {
            const size_t chunk = (npix + (size_t)c->world - 1) / (size_t)c->world;
            rc2 = comm_reduce_scatter_sum(c, rgbw, rgbw + (size_t)c->rank * chunk * 4, chunk * 4);     // in place
        }
        c->kev_end();
        return rc2;
    };
    // Fold the flags and - optimistically - merge the film behind the render: ONE host wait per render.  k_film_finalize
    // skips the merge when the (with a communicator: rank-summed) flag says that something went wrong somewhere.
    k_wh_any_flag<<<1, 32, 0, c->stream>>>(d_flags, (int)nb, d_err, d_flags + nb);
    c->stats.kernel_launches++;
    if (multi) {
        TR_CUDA(c, cudaMemsetAsync(d_flags + nb + 2, 0, 2 * sizeof(int), c->stream));
        if (comm_allreduce_sum_int(c, d_flags + nb, 2)) return 1;          // every rank learns whether ANY rank has to redo batches
        if (p2p) { if (film_sum_p2p(false, d_flags + nb)) return 1; }      // (the flag all-reduce is the opening barrier)
        else if (film_sum()) return 1;
    }
    if (f1 > f0 && !(multi && p2p)) {
        if (c->film_upload_pending) { TR_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_copy, 0)); c->film_upload_pending = false; }
        k_film_finalize<<<persistent_grid(c, 4), 256, 0, c->stream>>>(L.film_rgbw + f0, (float4*)film_dev + f0, (int)(f1 - f0), d_flags + nb);
        c->stats.kernel_launches++;
    }
    TR_CUDA(c, cudaEventRecord(c->ev1, c->stream));
    std::vector<int> h_flags((size_t)nb + 2, 0);
    TR_CUDA(c, cudaMemcpyAsync(h_flags.data(), d_flags, (size_t)(nb + 2) * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(c, cudaStreamSynchronize(c->stream));
    c->kev_collect();
    if (h_flags[(size_t)nb + 1]) {                              // (rank-summed: every rank fails together)
        cudaMemsetAsync(d_err, 0, sizeof(int), c->stream);
        return c->fail("traversal stack overflow (more than 64 pending nodes; the reference would throw a BoundsError, bvh.jl:222)");
    }
    if (h_flags[(size_t)nb]) {
        // A ray queue overflowed somewhere (rare: the queues hold cap_percent = 200 % of a batch): nothing has been merged.
        // Overflowed batches were not splatted: redo them in halves.  With a communicator the private film already went
        // through the (discarded) sum, so this rank's film is rebuilt from scratch, then summed and merged again.
        if (multi) {
            TR_CUDA(c, cudaMemsetAsync(L.film_rgbw, 0, npix_padded * sizeof(float4), c->stream));
            c->cur_lane = 0; c->cur_stream = c->stream;
        }
        for (long long bi = 0; bi < nb; ++bi) {
            if (!h_flags[bi]) { if (multi && run_batch(c, lane[0], b_begin[bi], b_count[bi], 1)) return 1; continue; }
            c->stats.queue_overflows++;
            const long long b = b_begin[bi], cnt = b_count[bi], half = cnt / 2 / per_tile * per_tile;
            if (cnt < 2 * per_tile) return c->fail("ray queue overflow that halving the batch cannot resolve");
            if (run_batch(c, lane[0], b, half, 1) || run_batch(c, lane[0], b + half, cnt - half, 1)) return 1;
        }
        if (multi && p2p) { if (film_sum_p2p(true, nullptr)) return 1; }
        else {
            if (multi && film_sum()) return 1;
            if (f1 > f0) {
                k_film_finalize<<<persistent_grid(c, 4), 256, 0, c->stream>>>(L.film_rgbw + f0, (float4*)film_dev + f0, (int)(f1 - f0), nullptr);
                c->stats.kernel_launches++;
            }
        }
        TR_CUDA(c, cudaEventRecord(c->ev1, c->stream));
        TR_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    float ms = 0.0f;
    cudaEventElapsedTime(&ms, c->ev0, c->ev1);
    c->stats.ms_total = ms;
    return 0;
}
