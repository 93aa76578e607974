// ref_render.cpp — CPU ORACLE (test infrastructure only): camera, film, Whitted and SPPM integrators.
// Follows src/camera/perspective.jl:85-114, src/film.jl:68-73,120-193, src/integrators/sampler.jl:12-199,
// src/integrators/sppm.jl:132-569, src/sampler/sampling.jl:3-76, src/sampler/primes.jl.
// The reference parallelises with Threads.@threads over 16x16 tiles and over photons; so does this file.
#include <algorithm>
#include <atomic>
#include <mutex>
#include <thread>

#include "ref_shading.hpp"

namespace ref {

// ---------------------------------------------------------------- camera
static Ray generate_ray(const trace_camera& c, float fx, float fy, float lu, float lv, float tu) {   // perspective.jl:85-114
    V3 pc = xf_point(c.raster_to_camera, V3(fx, fy, 0.0f));
    Ray r; r.o = V3(0.0f); r.d = normalize(pc); r.t_max = INF_F;
    if (c.lens_radius > 0.0f) {
        float lx, ly;
        concentric_sample_disk(lu, lv, lx, ly);
        lx = c.lens_radius * lx; ly = c.lens_radius * ly;
        float t = c.focal_distance / r.d.z;
        V3 pf = r.o + r.d * t;
        r.o = V3(lx, ly, 0.0f);
        r.d = normalize(pf - r.o);
    }
    r.time = (1.0f - tu) * c.shutter_open + tu * c.shutter_close;      // lerp, bounds.jl:122
    r.o = xf_point(c.camera_to_world, r.o);
    r.d = normalize(xf_vector(c.camera_to_world, r.d));
    return r;
}

// ---------------------------------------------------------------- film
struct TileBounds { int x0, y0, x1, y1; };

static void sample_bounds(const trace_film_desc& f, int& x0, int& y0, int& x1, int& y1) {   // film.jl:68-73
    x0 = (int)floorf((float)f.crop_x0 + 0.5f - f.filter_radius[0]);
    y0 = (int)floorf((float)f.crop_y0 + 0.5f - f.filter_radius[1]);
    x1 = (int)ceilf((float)f.crop_x1 - 0.5f + f.filter_radius[0]);
    y1 = (int)ceilf((float)f.crop_y1 - 0.5f + f.filter_radius[1]);
}
static TileBounds film_tile_bounds(const trace_film_desc& f, int sx0, int sy0, int sx1, int sy1) {   // film.jl:120-125
    TileBounds t;
    t.x0 = std::max((int)ceilf((float)sx0 - 0.5f - f.filter_radius[0]), f.crop_x0);
    t.y0 = std::max((int)ceilf((float)sy0 - 0.5f - f.filter_radius[1]), f.crop_y0);
    t.x1 = std::min((int)(floorf((float)sx1 - 0.5f + f.filter_radius[0]) + 1.0f), f.crop_x1);
    t.y1 = std::min((int)(floorf((float)sy1 - 0.5f + f.filter_radius[1]) + 1.0f), f.crop_y1);
    return t;
}
// add_sample!, film.jl:134-164. contrib/weight arrays are (ty1-ty0+1) x (tx1-tx0+1), row-major [y][x].
static void add_sample(const trace_film_desc& f, const TileBounds& tb, float px, float py, RGB L, float sw,
                       float* contrib, float* wsum) {
    float dx = px - 0.5f, dy = py - 0.5f;
    float p0x = ceilf(dx - f.filter_radius[0]), p0y = ceilf(dy - f.filter_radius[1]);
    float p1x = floorf(dx + f.filter_radius[0]) + 1.0f, p1y = floorf(dy + f.filter_radius[1]) + 1.0f;
    p0x = std::max(p0x, std::max((float)tb.x0, 1.0f)); p0y = std::max(p0y, std::max((float)tb.y0, 1.0f));
    p1x = std::min(p1x, (float)tb.x1); p1y = std::min(p1y, (float)tb.y1);
    float irx = 1.0f / f.filter_radius[0], iry = 1.0f / f.filter_radius[1];
    int tw = tb.x1 - tb.x0 + 1;
    for (float y = p0y; y <= p1y; y += 1.0f) {
        float fyv = fabsf((y - dy) * iry * 16.0f);
        int oy = (int)jl_clamp(floorf(fyv), 1.0f, 16.0f);
        for (float x = p0x; x <= p1x; x += 1.0f) {
            float fxv = fabsf((x - dx) * irx * 16.0f);
            int ox = (int)jl_clamp(ceilf(fxv), 1.0f, 16.0f);
            float w = f.filter_table[(oy - 1) * 16 + (ox - 1)];
            int ix = (int)x - tb.x0, iy = (int)y - tb.y0;
            float* c = contrib + 3 * ((size_t)iy * tw + ix);
            RGB add = (L * sw) * w;
            c[0] += add.r; c[1] += add.g; c[2] += add.b;
            wsum[(size_t)iy * tw + ix] += w;
        }
    }
}

// ---------------------------------------------------------------- Whitted, integrators/sampler.jl:58-199
struct RayCount { uint64_t closest = 0, shadow = 0; };

static RGB whitted_li(const Scene& s, Ray ray, int depth, int max_depth, RayCount& rc) {
    RGB l(0.0f);
    Hit hit;
    rc.closest++;
    if (!intersect_closest(s, ray, hit, 0, nullptr)) return l;            // le(light, ray) == 0, light.jl:41
    SurfaceInteraction si;
    build_interaction(s, ray, hit, si);
    V3 n = si.ns, wo = si.wo;
    BSDF bsdf;
    compute_scattering(s, si, false, bsdf);
    for (const trace_light& light : s.lights) {
        RGB li; V3 wi, lp; float pdf;
        sample_li(light, si.p, li, wi, pdf, lp);
        if (is_black(li) || pdf == 0.0f) continue;
        RGB f = bsdf_f(bsdf, wo, wi);
        if (!is_black(f)) {
            Ray sr = shadow_ray(si.p, lp);
            rc.shadow++;
            if (!intersect_any(s, sr, 0, nullptr)) l = l + (f * li) * fabsf(dot(wi, n)) / pdf;
        }
    }
    if (depth + 1 <= max_depth) {
        for (int pass = 0; pass < 2; ++pass) {                              // specular_reflect, specular_transmit
            uint8_t type = (pass == 0 ? BSDF_REFLECTION : BSDF_TRANSMISSION) | BSDF_SPECULAR;
            BSDFSample bs = bsdf_sample_f(bsdf, wo, 0.5f, 0.5f, type);     // u is unused by the specular lobes
            V3 ns = si.ns;
            if (!(bs.pdf > 0.0f && !is_black(bs.f) && fabsf(dot(bs.wi, ns)) != 0.0f)) continue;
            Ray rd = spawn_ray_dir(si.p, bs.wi);
            RGB child = whitted_li(s, rd, depth + 1, max_depth, rc);
            l = l + (bs.f * child) * fabsf(dot(bs.wi, ns)) / bs.pdf;
        }
    }
    return l;
}

}  // namespace ref

using namespace ref;

static int render_whitted_impl(const ref_scene* rs, const trace_camera* cam, const trace_film_desc* film, int spp,
                               int max_depth, uint64_t seed, float* film_xyzw, int n_threads, int64_t max_tiles,
                               uint64_t* ray_counters, const int64_t* tile_list, int64_t n_tile_list);

extern "C" int ref_render_whitted(const ref_scene* rs, const trace_camera* cam, const trace_film_desc* film, int spp,
                                  int max_depth, uint64_t seed, float* film_xyzw, int n_threads, int64_t max_tiles,
                                  uint64_t* ray_counters) {
    return render_whitted_impl(rs, cam, film, spp, max_depth, seed, film_xyzw, n_threads, max_tiles, ray_counters, nullptr, -1);
}
// explicit tile list (k = ty * n_tiles_x + tx): used to check the multi-GPU tile partition on CPU and to compare full-size
// films over one rank's share of the tiles
extern "C" int ref_render_whitted_tiles(const ref_scene* rs, const trace_camera* cam, const trace_film_desc* film, int spp,
                                        int max_depth, uint64_t seed, float* film_xyzw, const int64_t* tiles, int64_t n_tiles,
                                        int n_threads, uint64_t* ray_counters) {
    return render_whitted_impl(rs, cam, film, spp, max_depth, seed, film_xyzw, n_threads < 1 ? 1 : n_threads, 0, ray_counters, tiles, n_tiles);
}

static int render_whitted_impl(const ref_scene* rs, const trace_camera* cam, const trace_film_desc* film, int spp,
                               int max_depth, uint64_t seed, float* film_xyzw, int n_threads, int64_t max_tiles,
                               uint64_t* ray_counters, const int64_t* tile_list, int64_t n_tile_list) {
    const Scene& s = rs->s;
    int sx0, sy0, sx1, sy1;
    sample_bounds(*film, sx0, sy0, sx1, sy1);
    const int tile_size = 16;
    int width = (int)floorf(((float)(sx1 - sx0) + tile_size) / tile_size);   // sampler.jl:14-20
    int height = (int)floorf(((float)(sy1 - sy0) + tile_size) / tile_size);
    int64_t total = (int64_t)width * height;
    int sbw = sx1 - sx0 + 1;
    int fw = film->crop_x1 - film->crop_x0 + 1;
    std::vector<int64_t> tiles;
    if (n_tile_list >= 0) {
        for (int64_t j = 0; j < n_tile_list; ++j) if (tile_list[j] >= 0 && tile_list[j] < total) tiles.push_back(tile_list[j]);
    } else if (max_tiles > 0 && max_tiles < total) {
        for (int64_t j = 0; j < max_tiles; ++j) tiles.push_back(j * total / max_tiles);
    } else {
        for (int64_t k = 0; k < total; ++k) tiles.push_back(k);
    }
    std::atomic<int64_t> next(0);
    std::mutex merge_mutex;
    std::vector<RayCount> rcs(std::max(1, n_threads));
    auto worker = [&](int tid) {
        std::vector<float> contrib, wsum;
        for (;;) {
            int64_t j = next.fetch_add(1);
            if (j >= (int64_t)tiles.size()) break;
            int64_t k = tiles[j];
            int tx = (int)(k % width), ty = (int)(k / width);
            int bx0 = sx0 + tx * tile_size, by0 = sy0 + ty * tile_size;
            int bx1 = std::min(bx0 + tile_size - 1, sx1), by1 = std::min(by0 + tile_size - 1, sy1);
            TileBounds tb = film_tile_bounds(*film, bx0, by0, bx1, by1);
            int tw = tb.x1 - tb.x0 + 1, th = tb.y1 - tb.y0 + 1;
            if (tw <= 0 || th <= 0) continue;
            contrib.assign((size_t)tw * th * 3, 0.0f);
            wsum.assign((size_t)tw * th, 0.0f);
            for (int py = by0; py <= by1; ++py) for (int px = bx0; px <= bx1; ++px) {      // Bounds2 iteration, bounds.jl:39-47
                uint32_t pix = (uint32_t)((py - sy0) * sbw + (px - sx0));
                for (int sidx = 0; sidx < spp; ++sidx) {
                    float u0 = rng_uniform(seed, pix, sidx, 0), u1 = rng_uniform(seed, pix, sidx, 1);
                    float l0 = rng_uniform(seed, pix, sidx, 2), l1 = rng_uniform(seed, pix, sidx, 3);
                    float tu = rng_uniform(seed, pix, sidx, 4);
                    float fx = (float)px + u0, fy = (float)py + u1;
                    Ray ray = generate_ray(*cam, fx, fy, l0, l1, tu);
                    RGB l = whitted_li(s, ray, 1, max_depth, rcs[tid]);
                    if (has_nan(l)) l = RGB(0.0f);
                    add_sample(*film, tb, fx, fy, l, 1.0f, contrib.data(), wsum.data());
                }
            }
            std::lock_guard<std::mutex> g(merge_mutex);                                   // merge_film_tile!, film.jl:182-193
            for (int y = 0; y < th; ++y) for (int x = 0; x < tw; ++x) {
                float xyz[3];
                const float* c = &contrib[3 * ((size_t)y * tw + x)];
                rgb_to_xyz(RGB(c[0], c[1], c[2]), xyz);
                float* dst = film_xyzw + 4 * ((size_t)(tb.y0 + y - film->crop_y0) * fw + (tb.x0 + x - film->crop_x0));
                dst[0] += xyz[0]; dst[1] += xyz[1]; dst[2] += xyz[2];
                dst[3] += wsum[(size_t)y * tw + x];
            }
        }
    };
    if (n_threads <= 1) worker(0);
    else {
        std::vector<std::thread> th;
        for (int t = 0; t < n_threads; ++t) th.emplace_back(worker, t);
        for (auto& t : th) t.join();
    }
    if (ray_counters) {
        ray_counters[0] = ray_counters[1] = 0;
        for (auto& r : rcs) { ray_counters[0] += r.closest; ray_counters[1] += r.shadow; }
    }
    return 0;
}

// ---------------------------------------------------------------- Halton, sampling.jl:43-76
namespace ref {
// PRIMES (sampler/primes.jl): the 1023 odd primes 3 .. 8161; PRIMES[k] is the (k+1)-th prime.  Generated by a sieve.
static std::vector<int64_t> make_primes() {
    std::vector<char> composite(8200, 0);
    std::vector<int64_t> out;
    for (int i = 2; i < 8200 && out.size() < 1023; ++i) {
        if (composite[i]) continue;
        if (i > 2) out.push_back(i);
        for (int j = i * i; j < 8200; j += i) composite[j] = 1;
    }
    return out;
}
static const std::vector<int64_t> PRIMES_HEAD = make_primes();
static uint32_t reverse_bits32(uint32_t n) {
    n = (n << 16) | (n >> 16);
    n = ((n & 0x00ff00ffu) << 8) | ((n & 0xff00ff00u) >> 8);
    n = ((n & 0x0f0f0f0fu) << 4) | ((n & 0xf0f0f0f0u) >> 4);
    n = ((n & 0x33333333u) << 2) | ((n & 0xccccccccu) >> 2);
    return ((n & 0x55555555u) << 1) | ((n & 0xaaaaaaaau) >> 1);
}
static uint64_t reverse_bits64(uint64_t n) {
    uint64_t n0 = reverse_bits32((uint32_t)((n << 32) >> 32));
    uint64_t n1 = reverse_bits32((uint32_t)(n >> 32));
    return (n0 << 32) | n1;
}
float radical_inverse(int64_t base_index, uint64_t a) {
    if (base_index == 0) return (float)((double)reverse_bits64(a) * 5.4210108624275222e-20);
    int64_t base = PRIMES_HEAD.at((size_t)base_index - 1);            // PRIMES[base_index], 1-based
    float inv_base = 1.0f / (float)base;
    uint64_t reversed = 0;
    float inv_base_n = 1.0f;
    while (a > 0) {
        uint64_t next = (uint64_t)floor((double)a / (double)base);
        uint64_t digit = a - next * (uint64_t)base;
        reversed = reversed * (uint64_t)base + digit;
        inv_base_n *= inv_base;
        a = next;
    }
    return jl_min((float)reversed * inv_base_n, 1.0f);
}

// Distribution1D / sample_discrete, sampling.jl:3-41
struct Distribution1D {
    std::vector<float> func, cdf;
    float func_int;
    explicit Distribution1D(const std::vector<float>& f) : func(f) {
        size_t n = f.size();
        cdf.resize(n + 1);
        cdf[0] = 0.0f;
        for (size_t i = 1; i <= n; ++i) cdf[i] = cdf[i - 1] + func[i - 1] / (float)n;
        func_int = cdf[n];
        if (func_int == 0.0f) { for (size_t i = 1; i <= n; ++i) cdf[i] = (float)(i + 1) / (float)n; }
        else { for (size_t i = 1; i <= n; ++i) cdf[i] /= func_int; }
    }
    void sample(float u, int& off, float& pdf) const {
        int last = -1;
        for (int i = 0; i < (int)cdf.size(); ++i) if (cdf[i] <= u) last = i;
        int n = (int)func.size();
        off = std::min(std::max(last, 0), n - 1);
        pdf = func_int > 0.0f ? func[off] / (func_int * (float)n) : 0.0f;
    }
};

// ---------------------------------------------------------------- SPPM, integrators/sppm.jl
struct VisiblePoint { V3 p, wo; BSDF bsdf; bool has_bsdf; RGB beta; };
struct SPPMPixel {
    RGB Ld;
    std::atomic<float> phi[3];
    RGB tau;
    float radius;
    std::atomic<int64_t> M;
    double N;
    VisiblePoint vp;
};
static void atomic_add_f(std::atomic<float>& a, float v) {
    float old = a.load(std::memory_order_relaxed);
    while (!a.compare_exchange_weak(old, old + v, std::memory_order_relaxed)) {}
}

static RGB estimate_direct(const Scene& s, const SurfaceInteraction& si, const BSDF& bsdf, const trace_light& light,
                           RayCount& rc) {                                                       // sppm.jl:519-554
    uint8_t flags = BSDF_ALL & ~BSDF_SPECULAR;
    RGB Ld(0.0f);
    RGB Li; V3 wi, lp; float lpdf;
    sample_li(light, si.p, Li, wi, lpdf, lp);
    if (lpdf > 0.0f && !is_black(Li)) {
        RGB f = bsdf_f(bsdf, si.wo, wi, flags) * fabsf(dot(wi, si.ns));
        if (!is_black(f)) {
            Ray sr = shadow_ray(si.p, lp);
            rc.shadow++;
            if (intersect_any(s, sr, 0, nullptr)) Li = RGB(0.0f);
            if (!is_black(Li)) Ld = Ld + (f * Li) / lpdf;                                        // delta lights only
        }
    }
    return Ld;
}

static bool to_grid(V3 p, const B3& bounds, const int64_t res[3], int64_t out[3]) {            // sppm.jl:479-495
    V3 po = offset(bounds, p);
    int64_t g[3] = {(int64_t)floorf((float)res[0] * po.x), (int64_t)floorf((float)res[1] * po.y),
                    (int64_t)floorf((float)res[2] * po.z)};
    bool in = true;
    for (int i = 0; i < 3; ++i) {
        if (!(0 <= g[i] && g[i] < res[i])) in = false;
        out[i] = std::min(std::max(g[i], (int64_t)0), res[i] - 1);
    }
    return in;
}
static uint64_t grid_hash(uint64_t x, uint64_t y, uint64_t z, uint64_t size) {                   // sppm.jl:497-501 (0-based result)
    return ((x * 73856093ull) ^ (y * 19349663ull) ^ (z * 83492791ull)) % size;
}

}  // namespace ref

extern "C" int ref_render_sppm(const ref_scene* rs, const trace_camera* cam, const trace_film_desc* film, float r0,
                               int max_depth, int n_iterations, int64_t photons_per_iteration, uint64_t seed,
                               float* rgb_out, int n_threads, uint64_t* ray_counters) {
    const Scene& s = rs->s;
    const int W = film->crop_x1 - film->crop_x0 + 1, H = film->crop_y1 - film->crop_y0 + 1;   // inclusive_sides
    const uint64_t n_pixels = (uint64_t)W * H;
    if (photons_per_iteration <= 0)
        photons_per_iteration = (int64_t)(film->crop_x1 - film->crop_x0) * (film->crop_y1 - film->crop_y0);   // area(crop_bounds), Q22
    std::vector<SPPMPixel> pixels(n_pixels);
    for (auto& p : pixels) {
        p.Ld = RGB(0.0f); p.tau = RGB(0.0f); p.radius = r0; p.M = 0; p.N = 0.0;
        for (int k = 0; k < 3; ++k) p.phi[k] = 0.0f;
        p.vp.beta = RGB(0.0f); p.vp.has_bsdf = false;
    }
    const float gamma = 2.0f / 3.0f;
    std::vector<float> powers;
    for (const auto& l : s.lights) {
        if (l.kind == TRACE_LIGHT_DIRECTIONAL) return 2;      // no sample_le for DirectionalLight in the reference
        powers.push_back(to_Y(light_power(l)));
    }
    if (powers.empty()) return 1;
    Distribution1D light_distr(powers);
    const int tile_size = 16;
    int ntx = (int)floorf(((float)(film->crop_x1 - film->crop_x0) + tile_size) / tile_size);
    int nty = (int)floorf(((float)(film->crop_y1 - film->crop_y0) + tile_size) / tile_size);
    int nthr = std::max(1, n_threads);
    std::vector<RayCount> rcs(nthr);
    // CSR grid standing in for the linked lists (same multiset of (cell hash -> pixel) entries, Q10)
    std::vector<uint32_t> cell_start(n_pixels + 1), cell_items;

    for (int iteration = 1; iteration <= n_iterations; ++iteration) {
        // ---- _generate_visible_sppm_points!, sppm.jl:175-270
        {
            std::atomic<int> next(0);
            auto worker = [&](int tid) {
                RayCount& rc = rcs[tid];
                for (;;) {
                    int k = next.fetch_add(1);
                    if (k >= ntx * nty) break;
                    int tx = k % ntx, ty = k / ntx;
                    int bx0 = film->crop_x0 + tx * tile_size, by0 = film->crop_y0 + ty * tile_size;
                    int bx1 = std::min(bx0 + tile_size - 1, film->crop_x1), by1 = std::min(by0 + tile_size - 1, film->crop_y1);
                    for (int py = by0; py <= by1; ++py) for (int px = bx0; px <= bx1; ++px) {
                        uint32_t pix = (uint32_t)((py - film->crop_y0) * W + (px - film->crop_x0));
                        uint32_t it = (uint32_t)iteration;
                        float u0 = rng_uniform(seed, pix, it, 0), u1 = rng_uniform(seed, pix, it, 1);
                        float l0 = rng_uniform(seed, pix, it, 2), l1 = rng_uniform(seed, pix, it, 3);
                        float tu = rng_uniform(seed, pix, it, 4);
                        Ray ray = generate_ray(*cam, (float)px + u0, (float)py + u1, l0, l1, tu);
                        RGB beta(1.0f);
                        SPPMPixel& pixel = pixels[pix];
                        int depth = 1;
                        while (depth <= max_depth) {
                            uint32_t dim = 5 + 8 * (uint32_t)(depth - 1);
                            Hit hit;
                            rc.closest++;
                            if (!intersect_closest(s, ray, hit, 0, nullptr)) break;
                            SurfaceInteraction si;
                            build_interaction(s, ray, hit, si);
                            BSDF bsdf;
                            compute_scattering(s, si, true, bsdf);
                            V3 wo = -ray.d;
                            // uniform_sample_one_light, sppm.jl:503-517 (not multiplied by beta, Q8)
                            int nl = (int)s.lights.size();
                            float ul = rng_uniform(seed, pix, it, dim + 0);
                            int ln = std::max(1, std::min((int)ceilf(ul * (float)nl), nl));
                            float light_pdf = 1.0f / (float)nl;
                            pixel.Ld = pixel.Ld + estimate_direct(s, si, bsdf, s.lights[ln - 1], rc) / light_pdf;
                            bool is_diffuse = num_components(bsdf, BSDF_DIFFUSE | BSDF_REFLECTION | BSDF_TRANSMISSION) > 0;
                            bool is_glossy = num_components(bsdf, BSDF_GLOSSY | BSDF_REFLECTION | BSDF_TRANSMISSION) > 0;
                            if (is_diffuse || (is_glossy && depth == max_depth)) {
                                pixel.vp.p = si.p; pixel.vp.wo = wo; pixel.vp.bsdf = bsdf; pixel.vp.has_bsdf = true;
                                pixel.vp.beta = beta;
                                break;
                            }
                            if (depth == max_depth) { depth += 1; continue; }
                            BSDFSample bs = bsdf_sample_f(bsdf, wo, rng_uniform(seed, pix, it, dim + 5),
                                                          rng_uniform(seed, pix, it, dim + 6), BSDF_ALL);
                            if (bs.pdf == 0.0f || is_black(bs.f)) break;
                            beta = beta * (bs.f * fabsf(dot(bs.wi, si.ns)) / bs.pdf);
                            float by = to_Y(beta);
                            if (by < 0.25f) {
                                float cp = jl_min(1.0f, by);
                                if (rng_uniform(seed, pix, it, dim + 7) > cp) break;
                                beta = beta / cp;
                            }
                            ray = spawn_ray_dir(si.p, bs.wi);
                            depth += 1;
                        }
                    }
                }
            };
            if (nthr == 1) worker(0);
            else { std::vector<std::thread> th; for (int t = 0; t < nthr; ++t) th.emplace_back(worker, t); for (auto& t : th) t.join(); }
        }
        // ---- _populate_grid!, sppm.jl:278-318
        B3 grid_bounds;
        float max_radius = 0.0f;
        for (auto& p : pixels) {
            if (is_black(p.vp.beta)) continue;
            B3 e(p.vp.p - V3(p.radius), p.vp.p + V3(p.radius));
            grid_bounds = unite(grid_bounds, e);
            max_radius = jl_max(max_radius, p.radius);
        }
        V3 diag = diagonal(grid_bounds);
        float max_diag = jl_max(jl_max(diag.x, diag.y), diag.z);
        int64_t res[3] = {1, 1, 1};
        bool have_grid = max_radius > 0.0f && is_valid(grid_bounds);
        if (have_grid) {
            int64_t base = (int64_t)floorf(max_diag / max_radius);
            for (int i = 0; i < 3; ++i) res[i] = std::max((int64_t)1, (int64_t)floorf((float)base * diag[i] / max_diag));
        }
        std::fill(cell_start.begin(), cell_start.end(), 0u);
        cell_items.clear();
        if (have_grid) {
            for (int pass = 0; pass < 2; ++pass) {
                std::vector<uint32_t> cursor;
                if (pass == 1) {
                    uint32_t acc = 0;
                    for (uint64_t h = 0; h < n_pixels; ++h) { uint32_t c = cell_start[h]; cell_start[h] = acc; acc += c; }
                    cell_start[n_pixels] = acc;
                    cell_items.resize(acc);
                    cursor.assign(cell_start.begin(), cell_start.end() - 1);
                }
                for (uint64_t pi = 0; pi < n_pixels; ++pi) {
                    SPPMPixel& p = pixels[pi];
                    if (is_black(p.vp.beta)) continue;
                    int64_t lo[3], hi[3];
                    to_grid(p.vp.p - V3(p.radius), grid_bounds, res, lo);
                    to_grid(p.vp.p + V3(p.radius), grid_bounds, res, hi);
                    for (int64_t z = lo[2]; z <= hi[2]; ++z) for (int64_t y = lo[1]; y <= hi[1]; ++y) for (int64_t x = lo[0]; x <= hi[0]; ++x) {
                        uint64_t h = grid_hash((uint64_t)x, (uint64_t)y, (uint64_t)z, n_pixels);
                        if (pass == 0) cell_start[h]++; else cell_items[cursor[h]++] = (uint32_t)pi;
                    }
                }
            }
        }
        // ---- _trace_photons!, sppm.jl:320-436
        {
            uint64_t halton_base = (uint64_t)(iteration - 1) * (uint64_t)photons_per_iteration;
            std::atomic<int64_t> next(0);
            const int64_t CH = 4096;
            auto worker = [&](int tid) {
                RayCount& rc = rcs[tid];
                for (;;) {
                    int64_t c0 = next.fetch_add(CH);
                    if (c0 >= photons_per_iteration) break;
                    int64_t c1 = std::min(photons_per_iteration, c0 + CH);
                    for (int64_t photon = c0; photon < c1; ++photon) {
                        uint64_t hidx = halton_base + (uint64_t)photon;
                        int64_t hdim = 0;
                        float light_sample = radical_inverse(hdim, hidx);
                        hdim += 1;
                        int lnum; float light_pdf;
                        light_distr.sample(light_sample, lnum, light_pdf);
                        const trace_light& light = s.lights[lnum];
                        float ul0 = radical_inverse(hdim, hidx), ul1 = radical_inverse(hdim + 1, hidx);
                        hdim += 5;
                        LeSample le = sample_le(light, ul0, ul1);
                        if (le.pdf_pos == 0.0f || le.pdf_dir == 0.0f || is_black(le.le)) continue;
                        Ray pray = le.ray;
                        RGB beta = (fabsf(dot(le.n, pray.d)) * le.le) / (light_pdf * le.pdf_pos * le.pdf_dir);
                        if (is_black(beta)) continue;
                        float beta_y = to_Y(beta);
                        int depth = 1;
                        while (depth <= max_depth) {
                            Hit hit;
                            rc.closest++;
                            if (!intersect_closest(s, pray, hit, 0, nullptr)) break;
                            SurfaceInteraction si;
                            build_interaction(s, pray, hit, si);
                            if (depth > 1 && have_grid) {
                                int64_t gi[3];
                                if (to_grid(si.p, grid_bounds, res, gi)) {
                                    uint64_t h = grid_hash((uint64_t)gi[0], (uint64_t)gi[1], (uint64_t)gi[2], n_pixels);
                                    for (uint32_t e = cell_start[h]; e < cell_start[h + 1]; ++e) {
                                        SPPMPixel& px = pixels[cell_items[e]];
                                        V3 dd = px.vp.p - si.p;
                                        if (dot(dd, dd) > px.radius * px.radius) continue;
                                        RGB phi = beta * bsdf_f(px.vp.bsdf, px.vp.wo, -pray.d);
                                        atomic_add_f(px.phi[0], phi.r); atomic_add_f(px.phi[1], phi.g); atomic_add_f(px.phi[2], phi.b);
                                        px.M.fetch_add(1, std::memory_order_relaxed);
                                    }
                                }
                            }
                            BSDF bsdf;
                            compute_scattering(s, si, true, bsdf);
                            float b0 = radical_inverse(hdim, hidx), b1 = radical_inverse(hdim + 1, hidx);
                            hdim += 2;
                            BSDFSample bs = bsdf_sample_f(bsdf, -pray.d, b0, b1, BSDF_ALL);
                            if (is_black(bs.f) || bs.pdf == 0.0f) break;
                            RGB beta_new = ((beta * bs.f) * fabsf(dot(bs.wi, si.ns))) / bs.pdf;
                            float q = jl_max(0.0f, 1.0f - to_Y(beta_new) / beta_y);
                            if (radical_inverse(hdim, hidx) < q) { hdim += 1; break; }
                            hdim += 1;                                                    // beta is NOT updated (Q7)
                            pray = spawn_ray_dir(si.p, bs.wi);
                            depth += 1;
                        }
                    }
                }
            };
            if (nthr == 1) worker(0);
            else { std::vector<std::thread> th; for (int t = 0; t < nthr; ++t) th.emplace_back(worker, t); for (auto& t : th) t.join(); }
        }
        // ---- _update_pixels!, sppm.jl:438-459
        for (auto& p : pixels) {
            int64_t M = p.M.load();
            if (M > 0) {
                RGB phi(p.phi[0].load(), p.phi[1].load(), p.phi[2].load());
                double N_new = p.N + (double)(gamma * (float)M);
                double radius_new = (double)p.radius * sqrt(N_new / (p.N + (double)M));
                double ratio = radius_new / (double)p.radius;
                double r2 = ratio * ratio;
                RGB ts = p.tau + phi;
                p.tau = RGB((float)((double)ts.r * r2), (float)((double)ts.g * r2), (float)((double)ts.b * r2));
                p.radius = (float)radius_new;
                p.N = N_new;
                for (int k = 0; k < 3; ++k) p.phi[k] = 0.0f;
                p.M = 0;
            }
            p.vp.beta = RGB(0.0f);
            p.vp.has_bsdf = false;
        }
    }
    // ---- _sppm_to_image, sppm.jl:461-472
    double Np = (double)n_iterations * (double)photons_per_iteration * 3.141592653589793;
    for (uint64_t i = 0; i < n_pixels; ++i) {
        const SPPMPixel& p = pixels[i];
        RGB a = p.Ld / (float)n_iterations;
        double den = Np * (double)(p.radius * p.radius);
        RGB b((float)((double)p.tau.r / den), (float)((double)p.tau.g / den), (float)((double)p.tau.b / den));
        RGB c = a + b;
        rgb_out[3 * i] = c.r; rgb_out[3 * i + 1] = c.g; rgb_out[3 * i + 2] = c.b;
    }
    if (ray_counters) {
        ray_counters[0] = ray_counters[1] = 0;
        for (auto& r : rcs) { ray_counters[0] += r.closest; ray_counters[1] += r.shadow; }
    }
    return 0;
}

// ---------------------------------------------------------------- unit-level entry points
extern "C" float ref_fresnel_dielectric(float c, float ei, float et) { return fresnel_dielectric(c, ei, et); }
extern "C" float ref_radical_inverse(int64_t b, uint64_t a) { return radical_inverse(b, a); }
extern "C" float ref_roughness_to_alpha(float r) { return roughness_to_alpha(r); }
extern "C" float ref_rng(uint64_t seed, uint32_t a, uint32_t b, uint32_t c) { return rng_uniform(seed, a, b, c); }
static float sinc_f(float x) {                                           // filter.jl:12-17
    x = fabsf(x);
    if (x < 1e-5f) return 1.0f;
    x *= PI_F;
    return sinf(x) / x;
}
static float windowed_sinc(float x, float r, float tau) {                // filter.jl:19-23
    x = fabsf(x);
    if (x > r) return 0.0f;
    return sinc_f(x) * sinc_f(x / tau);
}
extern "C" float ref_lanczos(float px, float py, float rx, float ry, float tau) {
    return windowed_sinc(px, rx, tau) * windowed_sinc(py, ry, tau);
}
static void put_sample(const LobeSample& s, float out[8]) {
    out[0] = s.wi.x; out[1] = s.wi.y; out[2] = s.wi.z; out[3] = s.pdf;
    out[4] = s.f.r; out[5] = s.f.g; out[6] = s.f.b; out[7] = (float)s.sampled_type;
}
extern "C" int ref_fresnel_specular_sample(const float r[3], const float t[3], float ea, float eb, const float wo[3],
                                           const float u[2], float out[8]) {
    Lobe l = mk_lobe(L_FRESNEL_SPEC, BSDF_SPECULAR | BSDF_TRANSMISSION | BSDF_REFLECTION);
    l.r = RGB(r[0], r[1], r[2]); l.t = RGB(t[0], t[1], t[2]); l.eta_a = ea; l.eta_b = eb;
    put_sample(lobe_sample(l, V3(wo[0], wo[1], wo[2]), u[0], u[1]), out);
    return 0;
}
extern "C" int ref_microfacet_reflection_sample(const float r[3], float ax, float ay, int fk, float ei, float et,
                                                const float wo[3], const float u[2], float out[8]) {
    Lobe l = mk_lobe(L_MICRO_REFL, BSDF_REFLECTION | BSDF_GLOSSY);
    l.r = RGB(r[0], r[1], r[2]); l.fresnel = fk; l.fi = ei; l.ft = et;
    tr_alphas(l, ax, ay);
    put_sample(lobe_sample(l, V3(wo[0], wo[1], wo[2]), u[0], u[1]), out);
    return 0;
}
extern "C" int ref_microfacet_transmission_sample(const float t[3], float ax, float ay, float ea, float eb,
                                                  const float wo[3], const float u[2], float out[8]) {
    Lobe l = mk_lobe(L_MICRO_TRANS, BSDF_TRANSMISSION | BSDF_GLOSSY);          // microfacet.jl:261-278
    l.t = RGB(t[0], t[1], t[2]); l.eta_a = ea; l.eta_b = eb; l.fresnel = 1; l.fi = ea; l.ft = eb;
    tr_alphas(l, ax, ay);
    put_sample(lobe_sample(l, V3(wo[0], wo[1], wo[2]), u[0], u[1]), out);
    return 0;
}
static void canonical_bsdf(const trace_material* m, int mode, BSDF& b) {
    SurfaceInteraction si;
    si.p = V3(0.0f); si.wo = V3(0, 0, 1); si.ng = V3(0, 0, 1); si.ns = V3(0, 0, 1); si.sh_dpdu = V3(1, 0, 0);
    si.u = si.v = 0; si.prim = 0; si.material = 0;
    bsdf_init(b, si, 1.0f);
    material_lobes(*m, b, mode != 0);
}
extern "C" int ref_bsdf_f(const trace_material* m, int mode, const float wo[3], const float wi[3], int flags, float f[3]) {
    BSDF b; canonical_bsdf(m, mode, b);
    RGB v = bsdf_f(b, V3(wo[0], wo[1], wo[2]), V3(wi[0], wi[1], wi[2]), (uint8_t)flags);
    f[0] = v.r; f[1] = v.g; f[2] = v.b;
    return b.n;
}
extern "C" int ref_bsdf_sample(const trace_material* m, int mode, const float wo[3], const float u[2], int type, float out[8]) {
    BSDF b; canonical_bsdf(m, mode, b);
    BSDFSample s = bsdf_sample_f(b, V3(wo[0], wo[1], wo[2]), u[0], u[1], (uint8_t)type);
    out[0] = s.wi.x; out[1] = s.wi.y; out[2] = s.wi.z; out[3] = s.f.r; out[4] = s.f.g; out[5] = s.f.b;
    out[6] = s.pdf; out[7] = (float)s.type;
    return b.n;
}
// batched forms: q[i] = {material index, mode, flags (bsdf_f) or type (bsdf_sample)}; n_lobes[i] = the lobe count
extern "C" int ref_bsdf_f_batch(const trace_material* mats, int64_t n, const int32_t* q, const float* wo, const float* wi,
                                float* f, int32_t* n_lobes) {
    for (int64_t i = 0; i < n; ++i) n_lobes[i] = ref_bsdf_f(&mats[q[3 * i]], q[3 * i + 1], wo + 3 * i, wi + 3 * i, q[3 * i + 2], f + 3 * i);
    return 0;
}
extern "C" int ref_bsdf_sample_batch(const trace_material* mats, int64_t n, const int32_t* q, const float* wo, const float* u,
                                     float* out, int32_t* n_lobes) {
    for (int64_t i = 0; i < n; ++i) n_lobes[i] = ref_bsdf_sample(&mats[q[3 * i]], q[3 * i + 1], wo + 3 * i, u + 2 * i, q[3 * i + 2], out + 8 * i);
    return 0;
}
extern "C" int ref_film_tile_add_sample(const trace_film_desc* f, const int tbv[4], float px, float py, const float rgb[3],
                                        float* contrib, float* wsum) {
    TileBounds tb = {tbv[0], tbv[1], tbv[2], tbv[3]};
    add_sample(*f, tb, px, py, RGB(rgb[0], rgb[1], rgb[2]), 1.0f, contrib, wsum);
    return 0;
}
