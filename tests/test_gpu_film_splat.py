"""Every path of the Whitted film splat (whitted.cu k_wh_splat) against a float64 restatement of add_sample! and the
oracle's film (-m gpu): the per-sample path (spp not a multiple of 16), the grouped "packed" path (spp % 16 == 0, a
footprint window of at most 6 x 6) and the grouped "wide" path (a larger window: radius >= 2.5 or anisotropic radii),
with power-of-two and other spp (slot_to_pixel's shifts and its division), a film that is not a multiple of 16
tiles, a non-square crop window, the unfused primary path, many small batches on two lanes, and one rank's tile share.

The scene makes the film comparable almost exactly: a plane of sub-pixel checker triangles (albedo 0.9 / 0.05) that
fills the view, one preprocessed DirectionalLight and max_depth 1.  Each sample's radiance is then a few IEEE
operations on a closest hit that is bit-equal to the oracle's, so GPU and oracle agree sample by sample, and a
weight paired with a neighbouring sample's radiance changes the pixel visibly.

Bounds, per film pixel with n contributions of filter weights w_i and radiances L_i <= L_max, u = 2^-24:
- weight channel: the GPU sums the float32 weights in some order, so |W_gpu - sum w_i| <= (n - 1) u sum |w_i|
  against the float64 sum; asserted with (n + 1) u sum |w_i|.
- XYZ: both sides sum the products fl(L_i w_i) (error u each) in float32 in some order ((n - 1) u), the oracle per
  16 x 16 tile and then over the at most 4 tiles that overlap a pixel (3 u more), and convert with the 3-term row
  M_j of the RGB -> XYZ matrix (3 u).  So each side lies within (n + 6) u |M_j|_1 L_max sum |w_i| of the exact value,
  and |XYZ_gpu - XYZ_oracle| <= (2 n + 12) u |M_j|_1 L_max sum |w_i|.
- pixels no sample touches are exactly 0 on the GPU.
"""
import ctypes as C

import numpy as np
import pytest

import oracle_lib
import shading_cases as sc

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
M_ROW_L1 = np.array([0.412453 + 0.357580 + 0.180423, 0.212671 + 0.715160 + 0.072169, 0.019334 + 0.119193 + 0.950227])
LIGHT_I = 3.0
ALBEDO = (0.9, 0.05)
L_MAX = max(ALBEDO) / np.pi * LIGHT_I * (1 + 1e-6)       # f = albedo / pi, |cos| <= 1, Li = I (directional, pdf 1)


@pytest.fixture(scope="module")
def checker(T):
    """a 0.64 x 0.64 plane of 0.004-wide checker cells (2 triangles each; the view is about 0.5 wide, a pixel of the
    37 x 29 film about 3 cells) under a camera at height 10 looking down"""
    n, cell = 160, 0.004
    xs = (np.arange(n + 1) * cell - n * cell / 2).astype(np.float32)
    gx, gy = np.meshgrid(xs, xs)
    verts = np.stack([gx, gy, np.zeros_like(gx)], -1).reshape(-1, 3).astype(np.float32)
    i, j = np.meshgrid(np.arange(n), np.arange(n))
    v00 = (j * (n + 1) + i).ravel()
    v10, v01, v11 = v00 + 1, v00 + n + 1, v00 + n + 2
    parity = ((i + j) % 2).ravel()
    ident = T.ShapeCore(T.Transformation(), False)
    batches = []
    for par, albedo in zip((0, 1), ALBEDO):
        sel = parity == par
        tri = np.concatenate([np.stack([v00[sel], v10[sel], v11[sel]], 1), np.stack([v00[sel], v11[sel], v01[sel]], 1)])
        idx = (tri.ravel() + 1).astype(np.uint32)
        mesh = T.TriangleMesh(ident.object_to_world, len(tri), idx, len(verts), verts)
        mat = T.MatteMaterial(T.ConstantTexture(T.RGBSpectrum(albedo)), T.ConstantTexture(0.0))
        batches.append(T.PrimitiveBatch(T.TriangleSet(ident, mesh), mat))
    scene = T.Scene([], T.BVHAccel(batches, 1))
    sun = T.DirectionalLight(T.Transformation(), T.RGBSpectrum(LIGHT_I), [0.2, 0.3, 1.0])
    sun.preprocess(scene)
    scene.lights.append(sun)
    return scene


def camera(T, res, crop, radius):
    film = T.Film(res, T.Bounds2(crop[:2], crop[2:]), T.LanczosSincFilter(radius, 3.0), 1.0, 1.0, None)
    return T.PerspectiveCamera(T.look_at([0.05, 0.03, 10], [0, 0, 0], [0, 1, 0]), T.Bounds2([-1, -1], [1, 1]), 0, 1, 0, 1e6,
                               90.0, film)


def render_and_check(T, ctx, scene, cam_obj, spp, seed, tiles=None, label=""):
    flat = ctx.upload(scene)
    cam, fd = cam_obj.pod(), cam_obj.film.desc()
    gpu = np.zeros_like(cam_obj.film.pixels)
    ctx.check(ctx.lib.trace_render_whitted(ctx.h, C.byref(cam), C.byref(fd), spp, 1, C.c_uint64(seed), T._lib.ptr(gpu)))
    ref = np.zeros_like(gpu)
    osc = oracle_lib.OracleScene(flat)
    if tiles is None:
        osc.render_whitted(cam, fd, spp, 1, seed, ref)
    else:
        osc.render_whitted_tiles(cam, fd, spp, 1, seed, ref, tiles)
    fx, fy, tb = sc.whitted_film_samples(fd, spp, seed, tiles)
    ws, wabs, cnt = sc.restate_weights(fd, fx, fy, tb)
    touched = cnt > 0
    assert touched.any()
    assert np.all(gpu[~touched] == 0), f"{label}: {np.count_nonzero(np.any(gpu[~touched] != 0, -1))} untouched pixels are not 0"
    assert np.all(ref[~touched] == 0)
    werr = np.abs(gpu[..., 3].astype(np.float64) - ws)
    wbound = (cnt + 1) * U * wabs
    assert np.all(werr <= wbound), f"{label}: weight off by {(werr / np.maximum(wbound, 1e-300)).max():.3g} x the bound"
    xbound = (2 * cnt + 12)[..., None] * U * M_ROW_L1 * L_MAX * wabs[..., None]
    xerr = np.abs(gpu[..., :3].astype(np.float64) - ref[..., :3])
    assert np.all(xerr <= xbound), f"{label}: XYZ off by {(xerr / np.maximum(xbound, 1e-300)).max():.3g} x the bound"
    # the checker must make the film depend on which radiance meets which weight
    assert float(ref[..., 1].max()) > 0 and np.ptp(ref[touched][:, 1] / np.where(ws[touched] != 0, ws[touched], 1)) > 0.05
    print(f"splat {label}: {np.count_nonzero(touched)} pixels, weight err / bound {(werr / np.maximum(wbound, 1e-300)).max():.3g}, "
          f"XYZ err / bound {(xerr / np.maximum(xbound, 1e-300)).max():.3g}, max contributions {cnt.max()}")


RADII = [(0.5, 0.5), (1, 1), (1.5, 1.5), (2, 2), (2, 1), (2.5, 2.5), (4, 4), (4, 1.5)]


@pytest.mark.parametrize("radius", RADII)
@pytest.mark.parametrize("spp", [1, 3, 16, 48])
def test_splat_full_film(T, ctx, checker, radius, spp):
    """A 37 x 29 film (neither side a multiple of 16)."""
    render_and_check(T, ctx, checker, camera(T, [37, 29], (0, 0, 1, 1), radius), spp, 11 + spp, label=f"37x29 r{radius} spp{spp}")


def test_splat_spp32(T, ctx, checker):
    render_and_check(T, ctx, checker, camera(T, [37, 29], (0, 0, 1, 1), (1, 1)), 32, 5, label="37x29 r(1,1) spp32")


@pytest.mark.parametrize("radius,spp", [((1, 1), 16), ((4, 1.5), 16), ((2.5, 2.5), 48), ((1.5, 1.5), 3)])
def test_splat_crop_window(T, ctx, checker, radius, spp):
    """A non-square partial crop window: clipping to the crop and to pixel 1 of shifted tiles."""
    render_and_check(T, ctx, checker, camera(T, [64, 48], (0.1, 0.25, 0.8, 0.6), radius), spp, 7, label=f"crop r{radius} spp{spp}")


@pytest.mark.parametrize("radius,spp", [((1, 1), 3), ((2, 2), 16), ((4, 4), 16), ((2.5, 2.5), 48)])
def test_splat_unfused_primary(T, ctx, checker, radius, spp):
    """fuse_primary 0: k_wh_generate stores the film positions, the splat reads them back."""
    ctx.set_option("fuse_primary", 0)
    try:
        render_and_check(T, ctx, checker, camera(T, [37, 29], (0, 0, 1, 1), radius), spp, 3, label=f"unfused r{radius} spp{spp}")
    finally:
        ctx.set_option("fuse_primary", 1)


@pytest.mark.parametrize("radius", [(1.5, 1.5), (4, 1.5)])
def test_splat_many_batches_two_lanes(T, ctx, checker, radius):
    """Batches of 65 536 samples on two lanes: each batch and lane covers a dealt run of tiles."""
    ctx.set_option("batch", 65536)
    ctx.set_option("lanes", 2)
    try:
        render_and_check(T, ctx, checker, camera(T, [96, 80], (0, 0, 1, 1), radius), 48, 9, label=f"batches r{radius} spp48")
    finally:
        ctx.set_option("batch", 1 << 26)
        ctx.set_option("lanes", 12)


@pytest.mark.parametrize("radius,spp", [((1, 1), 16), ((2.5, 2.5), 16), ((2, 1), 3)])
def test_splat_rank_share(T, ctx, checker, radius, spp):
    """rank 3 of 8: only the tiles k % 8 == 3, against the oracle's render of the same tiles."""
    cam_obj = camera(T, [70, 50], (0, 0, 1, 1), radius)
    sx0, sy0, sx1, sy1 = sc.sample_bounds(cam_obj.film.desc())
    n_tiles = ((sx1 - sx0 + 16) // 16) * ((sy1 - sy0 + 16) // 16)
    tiles = np.arange(3, n_tiles, 8)
    ctx.set_option("world", 8)
    ctx.set_option("rank", 3)
    try:
        render_and_check(T, ctx, checker, cam_obj, spp, 13, tiles=tiles, label=f"rank 3/8 r{radius} spp{spp}")
    finally:
        ctx.set_option("rank", 0)
        ctx.set_option("world", 1)
