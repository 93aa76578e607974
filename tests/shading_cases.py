"""Inputs and host restatements shared by the call-by-call shading tests (test_gpu_shading_calls.py,
test_gpu_film_splat.py, test_shading_probe_host.py): a material set that reaches every lobe and packing branch, edge
sets of directions and sample values, the counter-based RNG in numpy, and add_sample! (film.jl:134-164) restated."""
import numpy as np

from trace_jl_b200 import _lib as tl

LB_REFLECTION, LB_TRANSMISSION, LB_DIFFUSE, LB_GLOSSY, LB_SPECULAR, LB_ALL = 1, 2, 4, 8, 16, 31
# flag sets: LB_ALL; the SPPM camera pass's non-specular set; Whitted's two specular passes; every lobe type alone
F_FLAGS = [LB_ALL, LB_ALL & ~LB_SPECULAR, LB_SPECULAR | LB_REFLECTION, LB_SPECULAR | LB_TRANSMISSION,
           LB_SPECULAR | LB_REFLECTION | LB_TRANSMISSION, LB_DIFFUSE | LB_REFLECTION, LB_GLOSSY | LB_REFLECTION,
           LB_GLOSSY | LB_TRANSMISSION, LB_REFLECTION, LB_TRANSMISSION]
# sample types: everything, specular only (both Whitted passes and their union), non-specular
S_TYPES = [LB_ALL, LB_SPECULAR | LB_REFLECTION, LB_SPECULAR | LB_TRANSMISSION, LB_SPECULAR | LB_REFLECTION | LB_TRANSMISSION,
           LB_ALL & ~LB_SPECULAR]


def materials():
    """trace_material records: every kind; sigma 0 / negative / 20 / 90 / 120; alpha at the 1e-3 clamp, very rough,
    anisotropic, remap on and off; glass eta 1.5, 1 / 1.5 and exactly 1; negative or zero spectra (dropped lobes, zero
    lobes)."""
    rows = []

    def add(kind, a, b=(0, 0, 0), eta=1.0, ru=0.0, rv=0.0, remap=0):
        rows.append((kind, a, b, eta, ru, rv, remap))

    M, MI, G, P = tl.MAT_MATTE, tl.MAT_MIRROR, tl.MAT_GLASS, tl.MAT_PLASTIC
    for sigma in (0.0, -5.0, 20.0, 90.0, 120.0):
        add(M, (0.8, 0.6, 0.4), ru=sigma)
    add(M, (-0.2, 0.0, 0.0), ru=20.0)                               # black after the clamp: no lobe
    add(M, (0.5, -1.0, 0.25), ru=0.0)                               # one clamped channel
    add(MI, (0.9, 0.8, 0.7))
    add(MI, (-1.0, -1.0, -1.0))
    for eta in (1.5, 1.0 / 1.5, 1.0):
        add(G, (1, 1, 1), (0.9, 0.9, 0.9), eta)                     # specular: FresnelSpecular (mode 1) or two lobes
        add(G, (1, 1, 1), (0.9, 0.8, 0.7), eta, 0.3, 0.05, 1)        # rough, anisotropic, remapped
        add(G, (0.8, 0.8, 0.8), (1, 1, 1), eta, 1e-5, 1e-5, 0)       # alpha clamped to 1e-3
        add(G, (1, 1, 1), (1, 1, 1), eta, 0.9, 0.9, 0)              # very rough
    add(G, (1, 1, 1), (-1, 0, 0), 1.5, 0.2, 0.35, 1)                 # transmission dropped
    add(G, (0, 0, 0), (0.9, 0.9, 0.9), 1.5, 0.2, 0.2, 0)             # reflection dropped
    add(G, (0, 0, 0), (0, -1, 0), 1.5)                               # no lobe
    add(G, (1, 1, 1), (1, 1, 1), 1.5, 0.0, 0.25, 0)                  # one roughness 0: not specular
    add(P, (0.3, 0.5, 0.3), (0.4, 0.4, 0.4), ru=0.15, remap=1)
    add(P, (0.3, 0.5, 0.3), (0.4, 0.4, 0.4), ru=1e-5)
    add(P, (0.3, 0.5, 0.3), (0.4, 0.4, 0.4), ru=0.8)
    add(P, (0.0, 0.0, 0.0), (0.4, 0.4, 0.4), ru=0.3)                 # glossy only
    add(P, (0.6, 0.6, 0.6), (-0.4, 0.0, 0.0), ru=0.3)                # diffuse only
    add(P, (0.0, 0.0, 0.0), (0.0, 0.0, 0.0), ru=0.3)                 # no lobe
    m = np.zeros(len(rows), tl.material_dtype)
    for i, (kind, a, b, eta, ru, rv, remap) in enumerate(rows):
        m[i] = (kind, a, b, eta, ru, rv, remap)
    return m


def _unit(v):
    v = np.asarray(v, np.float64)
    return (v / np.linalg.norm(v, axis=-1, keepdims=True)).astype(np.float32)


def edge_directions(rng):
    """Unit-ish directions where the lobes branch: z in {0, +-tiny, +-1e-4}, exact normal incidence, x = 0 or y = 0,
    lengths 1 +- 1e-6, and uniform ones."""
    tiny = np.float32(1e-30)
    out = [[0, 0, 1], [0, 0, -1], [1, 0, 0], [0, 1, 0], [-1, 0, 0], [0, -1, 0]]
    for z in (0.0, tiny, -tiny, 1e-4, -1e-4, 1e-7, -1e-7):
        for phi in (0.3, 1.9, 4.0):
            s = np.sqrt(max(0.0, 1.0 - z * z))
            out.append([s * np.cos(phi), s * np.sin(phi), z])
    for z in (0.9, -0.9, 0.2, -0.2, 0.99995, -0.99995):
        s = np.sqrt(1.0 - z * z)
        out += [[0.0, s, z], [s, 0.0, z], [0.0, -s, z], [-s, 0.0, z]]
    out = [np.asarray(v, np.float32) for v in out]
    u = _unit(rng.normal(size=(64, 3)))
    out += list(u)
    out += list((u[:16] * np.float32(1 + 1e-6)).astype(np.float32)) + list((u[16:32] * np.float32(1 - 1e-6)).astype(np.float32))
    return np.array(out, np.float32)


def bsdf_f_inputs(rng, n_uniform):
    """(wo, wi) pairs: every edge direction against every other, wi = mirror(wo), -wo and wo, pairs on opposite
    sides, directions past the critical angle of eta 1.5, and uniform pairs on the sphere."""
    e = edge_directions(rng)
    wo = np.repeat(e, len(e), 0)
    wi = np.tile(e, (len(e), 1))
    ws = [wo, np.concatenate([e, e, e])]
    wis = [wi, np.concatenate([e * np.float32([-1, -1, 1]), -e, e]).astype(np.float32)]
    a = _unit(rng.normal(size=(n_uniform, 3)))
    b = _unit(rng.normal(size=(n_uniform, 3)))
    ws.append(a); wis.append(b)
    opp = b.copy(); opp[:, 2] = -np.sign(a[:, 2]) * np.abs(opp[:, 2])
    ws.append(a); wis.append(opp)
    # grazing inside the denser medium: sin(theta) > 1 / 1.5
    z = rng.uniform(0.0, np.sqrt(1 - (1 / 1.5) ** 2), n_uniform // 4)
    phi = rng.uniform(0, 2 * np.pi, len(z))
    s = np.sqrt(1 - z * z)
    crit = np.stack([s * np.cos(phi), s * np.sin(phi), -z], 1).astype(np.float32)
    ws.append(crit); wis.append(_unit(rng.normal(size=crit.shape)))
    return np.concatenate(ws).astype(np.float32), np.concatenate(wis).astype(np.float32)


def sample_u(rng, n, max_components=2):
    """(u0, u1) with u0 = k / mc exactly, u1 = 0.5, 0 and 1 - 2^-24 among uniform values."""
    one_minus = np.float32(1 - 2.0 ** -24)
    edges = [0.0, 0.5, one_minus, 1.0 / 3, 2.0 / 3, 0.25, 0.75]
    for mc in range(1, max_components + 1):
        edges += [np.float32(k) / np.float32(mc) for k in range(mc + 1)]
    edges = np.array(edges, np.float32)
    uu = np.stack(np.meshgrid(edges, edges), -1).reshape(-1, 2)
    return np.concatenate([uu, rng.random((n, 2), dtype=np.float32)]).astype(np.float32)


# ---------------------------------------------------------------- RNG and add_sample!
def rng_uniform(seed, a, b, c):
    """DESIGN.md "RNG" (device_common.cuh rng_uniform / the oracle's ref_rng) on uint64 numpy arrays."""
    with np.errstate(over="ignore"):
        seed, a, b, c = (np.asarray(x).astype(np.uint64) for x in (seed, a, b, c))
        z = seed ^ (a * np.uint64(0x9E3779B97F4A7C15)) ^ (((b << np.uint64(32)) | c) * np.uint64(0xD1B54A32D192ED03))
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return (z >> np.uint64(40)).astype(np.float32) * np.float32(5.9604644775390625e-8)


def sample_bounds(fd):
    """get_sample_bounds (film.jl:68-73) in float32, as the oracle and ctx_device_film compute it"""
    f = np.float32
    rx, ry = f(fd.filter_radius[0]), f(fd.filter_radius[1])
    return (int(np.floor(f(fd.crop_x0) + f(0.5) - rx)), int(np.floor(f(fd.crop_y0) + f(0.5) - ry)),
            int(np.ceil(f(fd.crop_x1) - f(0.5) + rx)), int(np.ceil(f(fd.crop_y1) - f(0.5) + ry)))


def tile_bounds(fd, bx0, by0, bx1, by1):
    """FilmTile bounds of the sample block [bx0, bx1] x [by0, by1] (film.jl:120-125), float32 arithmetic; int arrays"""
    f = np.float32
    rx, ry = f(fd.filter_radius[0]), f(fd.filter_radius[1])
    x0 = np.maximum(np.ceil(np.asarray(bx0).astype(f) - f(0.5) - rx).astype(np.int64), fd.crop_x0)
    y0 = np.maximum(np.ceil(np.asarray(by0).astype(f) - f(0.5) - ry).astype(np.int64), fd.crop_y0)
    x1 = np.minimum((np.floor(np.asarray(bx1).astype(f) - f(0.5) + rx) + f(1)).astype(np.int64), fd.crop_x1)
    y1 = np.minimum((np.floor(np.asarray(by1).astype(f) - f(0.5) + ry) + f(1)).astype(np.int64), fd.crop_y1)
    return x0, y0, x1, y1


def add_sample_footprint(fd, tb, px, py):
    """add_sample! (film.jl:134-164) over n samples at film positions (px, py) (float32), each clipped to its tile
    bounds tb = (x0, y0, x1, y1) (int arrays): the footprint and the filter-table index in float32, exactly as the oracle
    computes them.  Yields (sample index, pixel x, pixel y, weight) arrays, one batch per footprint offset."""
    f = np.float32
    rx, ry = f(fd.filter_radius[0]), f(fd.filter_radius[1])
    table = np.frombuffer(bytes(fd.filter_table), np.float32)
    px, py = np.asarray(px, f), np.asarray(py, f)
    dx, dy = px - f(0.5), py - f(0.5)
    p0x = np.maximum(np.ceil(dx - rx), np.maximum(tb[0].astype(f), f(1)))
    p0y = np.maximum(np.ceil(dy - ry), np.maximum(tb[1].astype(f), f(1)))
    p1x = np.minimum(np.floor(dx + rx) + f(1), tb[2].astype(f))
    p1y = np.minimum(np.floor(dy + ry) + f(1), tb[3].astype(f))
    irx, iry = f(1) / rx, f(1) / ry
    span_x, span_y = int(np.ceil(2 * rx)) + 2, int(np.ceil(2 * ry)) + 2
    idx = np.arange(len(px))
    for j in range(span_y):
        y = p0y + f(j)
        oy = np.clip(np.floor(np.abs((y - dy) * iry * f(16))), f(1), f(16)).astype(np.int64)
        for k in range(span_x):
            x = p0x + f(k)
            m = (y <= p1y) & (x <= p1x)
            if not m.any():
                continue
            ox = np.clip(np.ceil(np.abs((x[m] - dx[m]) * irx * f(16))), f(1), f(16)).astype(np.int64)
            yield idx[m], x[m].astype(np.int64), y[m].astype(np.int64), table[(oy[m] - 1) * 16 + (ox - 1)]


def whitted_film_samples(fd, spp, seed, tiles=None):
    """Every camera sample of a Whitted render (integrators/sampler.jl:12-57, slot layout aside): film position
    (fx, fy) from the RNG dimensions 0 and 1 and the bounds of the sample's tile.  tiles: the 16 x 16 sample tiles
    rendered (k = ty * tiles_x + tx), default all."""
    sx0, sy0, sx1, sy1 = sample_bounds(fd)
    f = np.float32
    tiles_x = int(np.floor((f(sx1 - sx0) + f(16)) / f(16)))
    tiles_y = int(np.floor((f(sy1 - sy0) + f(16)) / f(16)))
    if tiles is None:
        tiles = np.arange(tiles_x * tiles_y)
    tiles = np.asarray(tiles, np.int64)
    ty, tx = tiles // tiles_x, tiles % tiles_x
    j = np.arange(256)
    px = (sx0 + tx[:, None] * 16 + (j % 16)[None]).ravel()
    py = (sy0 + ty[:, None] * 16 + (j // 16)[None]).ravel()
    bx0, by0 = np.repeat(sx0 + tx * 16, 256), np.repeat(sy0 + ty * 16, 256)
    keep = (px <= sx1) & (py <= sy1)
    px, py, bx0, by0 = px[keep], py[keep], bx0[keep], by0[keep]
    tb = tile_bounds(fd, bx0, by0, np.minimum(bx0 + 15, sx1), np.minimum(by0 + 15, sy1))
    pix = ((py - sy0) * (sx1 - sx0 + 1) + (px - sx0)).astype(np.uint64)
    s = np.arange(spp, dtype=np.uint64)
    pixr = np.repeat(pix, spp)
    sr = np.tile(s, len(pix))
    fx = px.astype(f).repeat(spp) + rng_uniform(seed, pixr, sr, 0)
    fy = py.astype(f).repeat(spp) + rng_uniform(seed, pixr, sr, 1)
    tbr = tuple(np.repeat(t, spp) for t in tb)
    return fx.astype(f), fy.astype(f), tbr


def restate_weights(fd, fx, fy, tb):
    """float64 sum of the filter weights per film pixel, their count and the sum of |w|: [h, w] arrays"""
    w, h = fd.crop_x1 - fd.crop_x0 + 1, fd.crop_y1 - fd.crop_y0 + 1
    ws, wabs, cnt = np.zeros(h * w), np.zeros(h * w), np.zeros(h * w, np.int64)
    for _, x, y, wt in add_sample_footprint(fd, tb, fx, fy):
        k = (y - fd.crop_y0) * w + (x - fd.crop_x0)
        ws += np.bincount(k, wt.astype(np.float64), h * w)
        wabs += np.bincount(k, np.abs(wt.astype(np.float64)), h * w)
        cnt += np.bincount(k, minlength=h * w)
    return ws.reshape(h, w), wabs.reshape(h, w), cnt.reshape(h, w)
