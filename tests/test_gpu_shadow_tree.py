"""The shadow tree (an LBVH built on the device at upload, DeviceScene::shadow_pairs) and the any-hit walk over it
(traverse.cuh, traverse_shadow): with option shadow_tree 1 every any-hit answer equals the reference tree's walk
(shadow_tree 0) bit for bit - on shadow rays like the renders', random rays, crafted rays that need the exact
check's fallback, after a refit - and renders are unchanged."""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

f32 = np.float32


@pytest.fixture(scope="module")
def sctx(T):
    c = T.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def tess1m(T):
    return T.scenes.tessellated(cells=600, stacks=266, slices=264, res=(1920, 1080),
                                window=((-50.0, -28.125), (50.0, 28.125)))


@pytest.fixture(scope="module")
def caustic(T):
    if not os.path.exists(T.scenes.ASSET_PLY):
        pytest.skip("asset missing")
    return T.scenes.caustic_glass()


def occluded_both(ctx, o, d, t):
    """(answers with the shadow tree, answers without, fallbacks taken)"""
    ctx.set_option("shadow_tree", 1)
    ctx.reset_stats()
    on = ctx.occluded(o, d, t)
    fb = ctx.stats()["shadow_fallbacks"]
    ctx.set_option("shadow_tree", 0)
    off = ctx.occluded(o, d, t)
    ctx.set_option("shadow_tree", 1)
    return on, off, fb


def shadow_rays(ctx, flat, n, seed):
    """rays from surface points (closest hits of random rays through the scene) towards the lights and random points,
    t_max = 1 - 1e-4 as a shadow ray's (Whitted / SPPM spawn them with the light at t = 1)"""
    rng = np.random.default_rng(seed)
    lo, hi = flat.nodes[0]["bmin"], flat.nodes[0]["bmax"]
    ext = (hi - lo).astype(f32)
    tgt = (lo + rng.random((n, 3), dtype=f32) * ext).astype(f32)
    o = (tgt + rng.normal(size=(n, 3)).astype(f32) * f32(0.6 * np.abs(ext).max())).astype(f32)
    prim, t, _ = ctx.intersect(o, (tgt - o).astype(f32))
    hit = prim != 0
    p = (o + (tgt - o) * t[:, None]).astype(f32)[hit]
    lights = np.asarray(flat.lights["position"], f32).reshape(-1, 3)
    if len(lights) == 0:
        lights = (f32(0.5) * (lo + hi) + ext * f32([0, 0.5, 0]))[None].astype(f32)
    to = lights[rng.integers(0, len(lights), len(p))]
    far = (lo + rng.random((len(p), 3), dtype=f32) * ext).astype(f32)
    to = np.where(rng.random((len(p), 1)) < 0.5, to, far).astype(f32)
    d = (to - p).astype(f32)
    return p, d, np.full(len(p), 1.0 - 1e-4, f32)


def random_rays(flat, n, seed):
    rng = np.random.default_rng(seed)
    lo, hi = flat.nodes[0]["bmin"], flat.nodes[0]["bmax"]
    ext = (hi - lo).astype(f32)
    tgt = (lo + rng.random((n, 3), dtype=f32) * ext).astype(f32)
    o = (tgt + rng.normal(size=(n, 3)).astype(f32) * f32(0.5 * np.abs(ext).max())).astype(f32)
    d = (tgt - o).astype(f32)
    t = np.where(rng.random(n) < 0.5, np.inf, rng.uniform(0.2, 1.5, n)).astype(f32)
    return o, d, t


def _agree_on_scene(ctx, scene, seed):
    flat = ctx.upload(scene)
    assert ctx.shadow_tree() is not None
    n = 1_100_000
    fams = {"shadow": shadow_rays(ctx, flat, 2 * n, seed), "random": random_rays(flat, n, seed + 1)}
    o, d, _ = fams["random"]
    fams["random_inf"] = (o, d, np.full(len(o), np.inf, f32))
    total_fb = 0
    for name, (o, d, t) in fams.items():
        assert len(o) >= 1_000_000, name
        on, off, fb = occluded_both(ctx, o, d, t)
        assert np.array_equal(on, off), f"{name}: {np.count_nonzero(on != off)} answers differ"
        assert 0.02 < on.mean() < 0.98 or name == "random_inf", f"{name}: occluded fraction {on.mean()}"
        total_fb += fb
    return total_fb


def test_occluded_agrees_tess1m(sctx, tess1m):
    _agree_on_scene(sctx, tess1m[0], 11)


def test_occluded_agrees_caustic(sctx, caustic):
    _agree_on_scene(sctx, caustic[0], 21)


def _mesh_scene(T, tris):
    tris = np.asarray(tris, f32).reshape(-1, 3, 3)
    mat = T.MatteMaterial(T.ConstantTexture(T.RGBSpectrum(0.7)), T.ConstantTexture(0.0))
    n = len(tris)
    mesh = T.create_triangle_mesh(T.ShapeCore(T.Transformation(), False), n, list(range(1, 3 * n + 1)), 3 * n,
                                  tris.reshape(-1, 3).tolist())
    return T.Scene([T.PointLight(T.translate([0.3, 5.0, 0.2]), T.RGBSpectrum(5.0))],
                   T.BVHAccel([T.GeometricPrimitive(m, mat) for m in mesh], 1))


def _grid_tris(k=8):
    """a k x k grid of quads in the plane z = 0 (shared edges and vertices; an axis-aligned zero-thickness layer), a
    tilted strip and a box's faces (shared box faces)"""
    out = []
    for i in range(k):
        for j in range(k):
            a, b, c, d = [i, j, 0], [i + 1, j, 0], [i + 1, j + 1, 0], [i, j + 1, 0]
            out += [[a, b, c], [a, c, d]]
    for i in range(k):
        out.append([[i, 0, 1], [i + 1, 0, 1.5], [i, k, 2]])
    cube = np.array([[0, 0, -2], [2, 0, -2], [2, 2, -2], [0, 2, -2], [0, 0, -1], [2, 0, -1], [2, 2, -1], [0, 2, -1]], f32)
    for f in ([0, 1, 2], [0, 2, 3], [4, 5, 6], [4, 6, 7], [0, 1, 5], [0, 5, 4], [3, 2, 6], [3, 6, 7], [0, 3, 7], [0, 7, 4],
              [1, 2, 6], [1, 6, 5]):
        out.append(cube[f].tolist())
    return np.array(out, f32)


def crafted_rays(k=8):
    """axis-parallel rays, rays through shared edges and vertices of the grid, rays in and grazing the z = 0 plane,
    rays grazing the cube's faces; finite and infinite t_max"""
    rng = np.random.default_rng(5)
    o, d = [], []
    pts = np.array([[i, j, 0] for i in range(k + 1) for j in range(k + 1)], f32)
    mids = np.concatenate([pts + [0.5, 0, 0], pts + [0, 0.5, 0], pts + [0.5, 0.5, 0]]).astype(f32)
    for p in np.concatenate([pts, mids]):
        for dz in (1.0, -1.0):
            o.append(p + [0, 0, 3 * dz]); d.append([0, 0, -dz])                    # axis-parallel through vertices / edges
            dd = rng.normal(size=3).astype(f32)
            dd[2] = -abs(dd[2]) * dz - 0.1 * dz
            o.append(p - 3 * dd); d.append(dd)                                        # oblique through the same points
        o.append(p + [-1, 0, 0]); d.append([1, 0, 0])                                 # in the plane, along an axis
        o.append(p + [-1, -1, 0]); d.append([1, 1, 0])                                # in the plane, diagonal
        o.append(p + [-1, -1, 1e-7]); d.append([1, 1, -1e-7])                         # grazing the plane
    for x in np.linspace(-0.5, 2.5, 25, dtype=f32):
        for y in (0.0, 2.0, 1.0):
            o.append([x, y, -3]); d.append([0, 0, 1])                                 # along the cube's faces
            o.append([x, y, -3]); d.append([1e-3, 0, 1])
            o.append([x - 3, y, -1]); d.append([1, 0, 0])
    o, d = np.array(o, f32), np.array(d, f32)
    o, d = np.concatenate([o, o]), np.concatenate([d, d])
    t = np.concatenate([np.full(len(o) // 2, np.inf, f32), np.full(len(o) // 2, 4.0, f32)])
    return o, d, t


def test_crafted_rays_reach_fallback_and_agree(T, sctx):
    scene = _mesh_scene(T, _grid_tris())
    sctx.upload(scene)
    assert sctx.shadow_tree() is not None
    o, d, t = crafted_rays()
    on, off, fb = occluded_both(sctx, o, d, t)
    assert np.array_equal(on, off), f"{np.count_nonzero(on != off)} of {len(on)} answers differ"
    assert 0 < on.mean() < 1
    assert fb > 0


def test_no_shadow_tree_for_spheres_and_nan(T, sctx):
    scene, _, _ = T.scenes.shadows(resolution=32)
    flat = sctx.upload(scene)
    assert sctx.shadow_tree() is None
    o, d, t = random_rays(flat, 20_000, 3)
    on, off, fb = occluded_both(sctx, o, d, t)
    assert np.array_equal(on, off) and fb == 0
    # a NaN vertex (the host builders refuse NaN bounds, so the flat is patched after the build, as a caller's
    # buffers could be): the device build refuses it and the scene keeps the reference walk only
    import copy
    scene = _mesh_scene(T, _grid_tris())
    flat = copy.copy(scene.flatten())
    flat.tri_vertices = flat.tri_vertices.copy()
    flat.tri_vertices[5, 1, 0] = np.nan
    bad = T.Scene(scene.lights, scene.aggregate)
    bad._flat = flat
    sctx.upload(bad)
    assert sctx.shadow_tree() is None
    o, d, t = crafted_rays()
    on, off, fb = occluded_both(sctx, o, d, t)
    assert np.array_equal(on, off) and fb == 0


def test_refit_answers_equal_fresh_upload(T, sctx):
    from test_refit_host import refit_flat, tess_small, wave
    scene = tess_small(T)[0]
    flat = sctx.upload(scene)
    o, d, t = random_rays(flat, 400_000, 8)
    new = wave(flat, 0.7, seed=3)
    sctx.refit(scene, new)
    sctx.set_option("shadow_tree", 1)
    sctx.reset_stats()
    got = sctx.occluded(o, d, t)
    fresh = T.Context(0)
    try:
        fs = T.Scene(scene.lights, scene.aggregate)
        fs._flat = refit_flat(flat, new)
        fresh.upload(fs)
        fresh.set_option("shadow_tree", 0)
        want = fresh.occluded(o, d, t)
        assert np.array_equal(got, want)
        # the refit shadow tree equals the one a fresh upload builds over the same topology's new boxes: same answers,
        # and the boxes of a refit with the uploaded vertices come back bit for bit
        fresh.set_option("shadow_tree", 1)
        assert np.array_equal(fresh.occluded(o, d, t), want)
    finally:
        fresh.close()
    a = T.Context(0)
    try:
        s2 = tess_small(T)[0]
        a.upload(s2)
        before = a.shadow_tree()
        a.refit(s2)
        assert before.tobytes() == a.shadow_tree().tobytes()
    finally:
        a.close()


def test_two_uploads_give_identical_buffers(T, caustic):
    a, b = T.Context(0), T.Context(0)
    try:
        a.upload(caustic[0])
        b.upload(caustic[0])
        pa, pb = a.shadow_tree(), b.shadow_tree()
        assert pa is not None and pa.tobytes() == pb.tobytes()
        n = len(caustic[0].flatten().prims)
        assert pa.shape == (n - 1, 16)
        refs = pa.view(np.uint32)[:, [6, 14]].reshape(-1)
        leaves = refs[refs >= 0x80000000] & 0x7FFFFFFF
        assert np.array_equal(np.sort(leaves), np.arange(n))                        # one leaf per primitive slot
        assert np.array_equal(np.sort(refs[refs < 0x80000000]), np.arange(1, n - 1))  # every pair but the root once
    finally:
        a.close()
        b.close()


def _whitted(ctx, camera, spp=2, depth=5, seed=9):
    cam, fd = camera.pod(), camera.film.desc()
    film = np.zeros_like(camera.film.pixels)
    ctx.check(ctx.lib.trace_render_whitted(ctx.h, C.byref(cam), C.byref(fd), spp, depth, C.c_uint64(seed),
                                           film.ctypes.data_as(C.c_void_p)))
    return film


def _sppm(T, ctx, camera, r0, depth, photons, iters=3):
    cam, fd = camera.pod(), camera.film.desc()
    h, w = camera.film.pixels.shape[:2]
    rgb = np.zeros((h, w, 3), f32)
    ctx.check(ctx.lib.trace_render_sppm(ctx.h, C.byref(cam), C.byref(fd), r0, depth, iters, photons, 0, C.c_uint64(3),
                                        C.cast(None, T._lib.SPPM_CB), None, rgb.ctypes.data_as(C.c_void_p)))
    return rgb


def same_image(a, b):
    """equal up to the order of the float atomicAdd splats (as tests/test_gpu_refit.py)"""
    return np.allclose(a, b, rtol=2e-5, atol=2e-6 * float(np.abs(b).max()))


def test_renders_identical_with_and_without(T, sctx, caustic):
    from test_refit_host import tess_small
    scene, camera, _ = tess_small(T)
    sctx.upload(scene)
    out = {}
    for v in (1, 0):
        sctx.set_option("shadow_tree", v)
        out[v] = _whitted(sctx, camera)
    sctx.set_option("shadow_tree", 1)
    assert float(out[1][..., :3].max()) > 0 and same_image(out[1], out[0])
    scene, camera, kw = caustic
    sctx.upload(scene)
    assert sctx.shadow_tree() is not None
    img = {}
    for v in (1, 0):
        sctx.set_option("shadow_tree", v)
        img[v] = _sppm(T, sctx, camera, float(kw["initial_search_radius"]), int(kw["max_depth"]), 100_000)
        out[v] = _whitted(sctx, camera)
    sctx.set_option("shadow_tree", 1)
    assert float(img[1].max()) > 0 and same_image(img[1], img[0])
    assert same_image(out[1], out[0])
