"""The closest-hit walk on the shadow tree (option hit_tree, traverse.cuh traverse_closest_tree): with the option on every
closest-hit answer (primitive, t, b0, b1) equals the reference tree's walk (hit_tree 0) bit for bit - on camera rays,
reflected and refracted rays, random rays with infinite and finite t_max (also just above and below a hit's t),
crafted rays that need the fallback, after a refit and on an attached mesh - and renders are unchanged."""
import numpy as np
import pytest

from test_gpu_shadow_tree import _grid_tris, _mesh_scene, _sppm, _whitted, crafted_rays, random_rays, same_image

pytestmark = pytest.mark.gpu

f32 = np.float32
N = 1_000_000


@pytest.fixture(scope="module")
def hctx(T):
    c = T.Context(0)
    yield c
    c.close()


def intersect_both(ctx, o, d, t):
    """(answers with the walk on the shadow tree, answers without, fallbacks taken); answers = (prim, t, b)"""
    ctx.set_option("hit_tree", 1)
    ctx.reset_stats()
    on = ctx.intersect(o, d, t)
    fb = ctx.stats()["hit_fallbacks"]
    ctx.set_option("hit_tree", 0)
    off = ctx.intersect(o, d, t)
    ctx.set_option("hit_tree", 1)
    return on, off, fb


def assert_same(on, off, what):
    (pa, ta, ba), (pb, tb, bb) = on, off
    bad = (pa != pb) | (ta.view(np.uint32) != tb.view(np.uint32)) | np.any(ba.view(np.uint32) != bb.view(np.uint32), axis=1)
    assert not bad.any(), f"{what}: {np.count_nonzero(bad)} of {len(pa)} answers differ"


def camera_rays(camera, n, seed):
    """pinhole rays through random raster positions of the camera (raster -> camera -> world, as the camera model)"""
    cam = camera.pod()
    r2c = np.array(cam.raster_to_camera, np.float64).reshape(4, 4)
    c2w = np.array(cam.camera_to_world, np.float64).reshape(4, 4)
    H, W = camera.film.pixels.shape[:2]
    rng = np.random.default_rng(seed)
    p = np.stack([rng.uniform(0, W, n), rng.uniform(0, H, n), np.zeros(n), np.ones(n)], 1) @ r2c.T
    p = p[:, :3] / p[:, 3:4]
    d = p / np.linalg.norm(p, axis=1, keepdims=True)
    o = np.broadcast_to(c2w[:3, 3], (n, 3))
    return o.astype(f32), (d @ c2w[:3, :3].T).astype(f32)


def secondary_rays(ctx, flat, o, d):
    """reflected and refracted (eta 1.5) rays from the closest hits of (o, d), starting exactly on the surface"""
    prim, t, _ = ctx.intersect(o, d)
    hit = prim != 0
    p = (o + d * t[:, None]).astype(f32)[hit]
    tri = flat.tri_vertices[np.minimum(prim[hit], len(flat.tri_vertices)) - 1].astype(np.float64)
    n = np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0])
    n /= np.maximum(np.linalg.norm(n, axis=1, keepdims=True), 1e-30)
    w = d[hit].astype(np.float64)
    w /= np.linalg.norm(w, axis=1, keepdims=True)
    c = -(w * n).sum(1, keepdims=True)
    n = np.where(c < 0, -n, n)
    c = np.abs(c)
    refl = w + 2 * c * n
    eta = 1 / 1.5
    k = np.maximum(1 - eta * eta * (1 - c * c), 0)
    refr = eta * w + (eta * c - np.sqrt(k)) * n
    return np.concatenate([p, p]), np.concatenate([refl, refr]).astype(f32)


def ray_families(ctx, flat, camera, n, seed):
    out = {}
    if camera is not None:
        o, d = camera_rays(camera, n, seed)
        out["camera"] = (o, d, np.full(n, np.inf, f32))
        so, sd = secondary_rays(ctx, flat, o, d)
        out["secondary"] = (so, sd, np.full(len(so), np.inf, f32))
    o, d, t = random_rays(flat, n, seed + 1)
    out["random_inf"] = (o, d, np.full(n, np.inf, f32))
    prim, th, _ = ctx.intersect(o, d)
    # finite t_max: random, and one float above / below / at the hit's t
    pick = np.random.default_rng(seed + 2).integers(0, 4, n)
    tf = np.where(pick == 0, t, np.where(pick == 1, np.nextafter(th, f32(np.inf)),
                                         np.where(pick == 2, np.nextafter(th, f32(0)), th))).astype(f32)
    tf = np.where((prim == 0) & (pick > 0), t, tf).astype(f32)
    out["random_finite"] = (o, d, tf)
    return out


def _agree(ctx, scene, camera, seed, n=N):
    flat = ctx.upload(scene)
    assert ctx.shadow_tree() is not None
    for name, (o, d, t) in ray_families(ctx, flat, camera, n, seed).items():
        on, off, fb = intersect_both(ctx, o, d, t)
        assert_same(on, off, name)
        assert (on[0] != 0).mean() > 0.05, name
        # a t_max at or just above a hit's t leaves no room for the band, and a secondary ray starting exactly on its
        # surface meets that triangle again at t ~ 0: those rays are built to take the fallback
        if name == "random_finite":
            assert fb > 0
        elif name != "secondary":
            assert fb < 1e-3 * len(o), (name, fb)


def test_hits_agree_tess1m(hctx, T):
    scene, camera, _ = T.scenes.tessellated(cells=600, stacks=266, slices=264, res=(1920, 1080),
                                            window=((-50.0, -28.125), (50.0, 28.125)))
    _agree(hctx, scene, camera, 31)


def test_hits_agree_caustic(hctx, T):
    import os
    if not os.path.exists(T.scenes.ASSET_PLY):
        pytest.skip("asset missing")
    scene, camera, _ = T.scenes.caustic_glass()
    _agree(hctx, scene, camera, 41)


def test_hits_agree_tess10m_sample(hctx, T):
    import bench
    scene, camera, _, _ = bench.build_scene(T, "tess-10M")
    _agree(hctx, scene, camera, 51, n=250_000)


def _tie_tris():
    """the grid of test_gpu_shadow_tree (shared edges and vertices, a tilted strip, a box), every grid triangle twice
    (duplicated coplanar triangles: the reference's first-visited one must win), and a copy of the grid one float
    above (z = 2^-149 and one ulp of 1) and one float below"""
    g = _grid_tris()
    grid = g[:128]
    up = grid.copy(); up[..., 2] = np.nextafter(f32(1), f32(2))
    up0 = grid.copy(); up0[..., 2] = np.nextafter(f32(0), f32(1))
    lo1 = grid.copy(); lo1[..., 2] = f32(1)
    return np.concatenate([g, grid, up0, lo1, up]).astype(f32)


def test_crafted_rays_reach_fallback_and_agree(T, hctx):
    hctx.upload(_mesh_scene(T, _tie_tris()))
    assert hctx.shadow_tree() is not None
    o, d, t = crafted_rays()
    # zero direction components and non-finite origins
    rng = np.random.default_rng(9)
    zo = rng.uniform(-1, 9, (3000, 3)).astype(f32)
    zd = rng.normal(size=(3000, 3)).astype(f32)
    zd[:1000, 0] = 0; zd[1000:2000, 1] = 0; zd[2000:, 2] = -0.0
    zo[::7] = [np.inf, 1, 1]
    zo[3::7] = [np.nan, 1, 1]
    o, d = np.concatenate([o, zo]), np.concatenate([d, zd])
    t = np.concatenate([t, np.where(rng.random(3000) < 0.5, np.inf, 5.0).astype(f32)])
    on, off, fb = intersect_both(hctx, o, d, t)
    assert_same(on, off, "crafted")
    assert (on[0] != 0).any()
    assert fb > 0


def test_after_refit(T, hctx):
    from test_refit_host import tess_small, wave
    scene = tess_small(T)[0]
    flat = hctx.upload(scene)
    o, d, t = random_rays(flat, 400_000, 8)
    hctx.refit(scene, wave(flat, 0.7, seed=3))
    assert hctx.shadow_tree() is not None
    on, off, _ = intersect_both(hctx, o, d, t)
    assert_same(on, off, "refit")
    assert (on[0] != 0).mean() > 0.05


def test_attached_mesh(T, hctx):
    from test_gpu_attach_mesh import split_case
    base, mesh, _ = split_case(T, "tess_small", 1)
    hctx.upload(T.CompositeScene(base, mesh))
    assert hctx.shadow_tree() is not None
    o, d, t = random_rays(base.flatten(), 400_000, 12)
    on, off, _ = intersect_both(hctx, o, d, t)
    assert_same(on, off, "attached mesh")
    assert (on[0] != 0).mean() > 0.05
    # a composed scene without a shadow tree (analytic spheres in the base) walks the reference tree only
    base, mesh, _ = split_case(T, "shadows", 1)
    hctx.upload(T.CompositeScene(base, mesh))
    assert hctx.shadow_tree() is None
    o, d, t = random_rays(base.flatten(), 100_000, 13)
    on, off, fb = intersect_both(hctx, o, d, t)
    assert_same(on, off, "no shadow tree")
    assert fb == 0


def test_renders_identical_with_and_without(T, hctx):
    import os
    from test_refit_host import tess_small
    scene, camera, _ = tess_small(T)
    hctx.upload(scene)
    out = {}
    for v in (1, 0):
        hctx.set_option("hit_tree", v)
        out[v] = _whitted(hctx, camera)
    hctx.set_option("hit_tree", 1)
    assert float(out[1][..., :3].max()) > 0 and same_image(out[1], out[0])
    if not os.path.exists(T.scenes.ASSET_PLY):
        return
    scene, camera, kw = T.scenes.caustic_glass()
    hctx.upload(scene)
    img = {}
    for v in (1, 0):
        hctx.set_option("hit_tree", v)
        img[v] = _sppm(T, hctx, camera, float(kw["initial_search_radius"]), int(kw["max_depth"]), 100_000)
        out[v] = _whitted(hctx, camera)
    hctx.set_option("hit_tree", 1)
    assert float(img[1].max()) > 0 and same_image(img[1], img[0])
    assert same_image(out[1], out[0])
    # the SPPM path kernels (option sppm_path) carry the walk as well
    hctx.set_option("sppm_path", 1)
    try:
        for v in (1, 0):
            hctx.set_option("hit_tree", v)
            img[v] = _sppm(T, hctx, camera, float(kw["initial_search_radius"]), int(kw["max_depth"]), 100_000)
    finally:
        hctx.set_option("hit_tree", 1)
        hctx.set_option("sppm_path", 0)
    assert float(img[1].max()) > 0 and same_image(img[1], img[0])


def test_count_nodes_modes(T, hctx):
    from test_refit_host import tess_small
    flat = hctx.upload(tess_small(T)[0])
    o, d, _ = random_rays(flat, 200_000, 4)
    counts = {}
    for mode in (1, 2):
        hctx.set_option("count_nodes", mode)
        hctx.reset_stats()
        hctx.intersect(o, d)
        counts[mode] = hctx.stats()["nodes_visited"]
        hctx.set_option("count_nodes", 0)
    assert counts[1] > 0 and counts[2] > 0 and counts[1] != counts[2]
    with pytest.raises(RuntimeError):
        hctx.set_option("count_nodes", 3)
