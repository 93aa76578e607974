"""Mesh attach (trace_scene_attach_mesh_device, csrc/upload_device.cu; CompositeScene + Context.upload).  Its contract:
the composed device scene is bit for bit the scene trace_scene_upload builds from D (tests/test_attach_mesh_host.py,
`compose_restate`), and its shadow tree is the composition of the two parts' own (`compose_shadow`).  Checked here
against D uploaded by hand in a second context: nodes, shadow tree, ray answers under both walks, images; then
sequences of attaches, refit, refusals, the shadow tree's depth rule, determinism and memory."""
import ctypes as C

import numpy as np
import pytest

from test_attach_mesh_host import compose_restate, compose_shadow
from test_gpu_device_upload import answers, host_scene, jl_bounds, ray_families, same_answers
from test_gpu_lbvh import deep_bounds, gpu_build, lbvh_restate, same_bits
from test_gpu_refit import same_image
from test_refit_host import wave

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dctx(T):
    c = T.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def hctx(T):
    c = T.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def sctx(T):
    c = T.Context(0)
    yield c
    c.close()


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda(0)


def split(T, scene, pick, m, builder):
    """(base Scene, DeviceMeshScene): the PrimitiveBatch aggregate.items[pick] becomes the mesh, the rest the base"""
    items = [p for _, p in scene.aggregate.items]
    batch = items[pick]
    base = T.Scene(scene.lights, T.BVHAccel(items[:pick] + items[pick + 1:], m, builder=builder))
    mesh, core = batch.triangles.mesh, batch.triangles.core
    v, tn = mesh.triangle_vertices(), mesh.triangle_normals()
    flags = np.full(len(v), (1 if core.flip else 0) | (2 if tn is not None else 0), np.uint8)
    return base, T.DeviceMeshScene([], _dev(v), [batch.material], None, None if tn is None else _dev(tn), _dev(flags),
                                   max_node_primitives=m)


def sphere_mesh(T, center, radius, stacks, slices, m=1, material=None):
    v, n, idx = T.scenes._uv_sphere(center, radius, stacks, slices)
    i = idx.astype(np.int64).reshape(-1, 3) - 1
    mat = material or T.MirrorMaterial(T.ConstantTexture(T.RGBSpectrum(0.9)))
    light = T.PointLight(T.translate(np.array(center, np.float32) + np.float32(3 * radius)), T.RGBSpectrum(5.0))
    return T.DeviceMeshScene([light], _dev(v[i]), [mat], None, _dev(n[i]), _dev(np.full(len(i), 2, np.uint8)),
                             max_node_primitives=m)


def split_case(T, name, m):
    """(base, mesh, camera): tess_small / tess_1M without their mirror sphere, which becomes the mesh; the caustic floor
    with the glass PLY as the mesh; the shadows scene (analytic spheres) with a small sphere mesh"""
    if name == "shadows":
        scene, camera, _ = T.scenes.shadows(resolution=64)
        return scene, sphere_mesh(T, (0.5, 0.6, -2.5), 0.15, 10, 12, m), camera
    scene, camera = host_scene(T, name, m)
    base, mesh = split(T, scene, 0 if name == "caustic" else 2, m, "reference")
    return base, mesh, camera


def _host(t):
    return None if t is None else t.cpu().numpy()


def upload_d(T, ctx, base, mesh, base_nodes=None, base_vertices=None):
    """trace_scene_upload of D, made by hand: -> (D's nodes, prims).  `base_nodes` / `base_vertices`: the base's
    current ones (after a refit), default its flattening's"""
    flat = base.flatten()
    bn = flat.nodes if base_nodes is None else base_nodes
    bv = flat.tri_vertices if base_vertices is None else base_vertices
    mv, mn, mf = _host(mesh.vertices), _host(mesh.normals), _host(mesh.flags)
    n = len(mv)
    mids = np.zeros(n, np.uint32) if mesh.material_ids is None else _host(mesh.material_ids).astype(np.uint32)
    rc, mnodes, morder = gpu_build(jl_bounds(mv), mesh.max_node_primitives)
    assert rc == 0
    nodes, prims = compose_restate(bn, flat.prims, len(flat.tri_vertices), flat.n_materials, mnodes, morder, mids)
    if mn is None:
        mn = np.zeros_like(mv)
    mf = np.zeros(n, np.uint8) if mf is None else mf
    if mesh.normals is None:
        mf = mf & ~np.uint8(2)
    v = np.ascontiguousarray(np.concatenate([bv, mv]), np.float32)
    nrm = np.ascontiguousarray(np.concatenate([flat.tri_normals, mn]), np.float32)
    f = np.ascontiguousarray(np.concatenate([flat.tri_flags, mf]), np.uint8)
    _, (mmats, mlights) = mesh.desc(0)
    mats = np.ascontiguousarray(np.concatenate([flat.materials_pod[:flat.n_materials], mmats[:len(mesh.materials)]]))
    lights = np.ascontiguousarray(np.concatenate([flat.lights, mlights]))
    d = T._lib.SceneDesc()
    d.n_nodes, d.nodes = len(nodes), T._lib.ptr(nodes)
    d.n_prims, d.prims = len(prims), T._lib.ptr(prims)
    d.n_tris, d.tri_vertices, d.tri_normals, d.tri_flags = len(v), T._lib.ptr(v), T._lib.ptr(nrm), T._lib.ptr(f)
    d.n_spheres, d.spheres = len(flat.spheres), T._lib.ptr(flat.spheres)
    d.n_materials, d.materials = len(mats), T._lib.ptr(mats)
    d.n_lights, d.lights = len(lights), T._lib.ptr(lights)
    ctx.check(ctx.lib.trace_scene_upload(ctx.h, C.byref(d)))
    ctx._scene, ctx._n_nodes, ctx._base, ctx._mesh = object(), len(nodes), None, None   # (never cached)
    return nodes, prims


def expected_shadow(sctx, base, mesh, axis):
    """the composition of the two parts' own shadow trees, each uploaded alone (None when a part has none)"""
    sctx.upload(base)
    bs = sctx.shadow_tree()
    sctx.upload(mesh)
    ms = sctx.shadow_tree()
    if bs is None or ms is None:
        return None
    return compose_shadow(bs, ms, axis)


def both_walks(ctxs, rays):
    out = []
    for walk in (0, 1):
        for c in ctxs:
            c.set_option("walk", walk)
        out.append([answers(c, rays) for c in ctxs])
    for c in ctxs:
        c.set_option("walk", 1)
    return out


CASES = [("tess_small", 1), ("caustic", 1), ("caustic", 4), ("tess_1M", 1), ("shadows", 1)]


@pytest.mark.parametrize("name, m", CASES)
def test_exact_contract(T, dctx, hctx, sctx, name, m):
    base, mesh, camera = split_case(T, name, m)
    cs = T.CompositeScene(base, mesh)
    assert dctx.upload(cs) is cs
    nodes = dctx.scene_nodes()
    dn, _ = upload_d(T, hctx, base, mesh)
    assert same_bits(nodes, hctx.scene_nodes()) and same_bits(nodes, dn)
    sh = expected_shadow(sctx, base, mesh, int(dn[0]["meta"]) >> 30)
    if name == "shadows":
        assert sh is None and dctx.shadow_tree() is None
    else:
        assert sh is not None and same_bits(dctx.shadow_tree(), sh)
    n = 1_000_000 if name in ("tess_1M", "caustic") else 200_000
    rays = ray_families(T, cs, camera, n, seed=11 + m)
    for a, b in both_walks([dctx, hctx], rays):
        assert (a[1][0] != 0).mean() > 0.02 and a[1][3].mean() > 0.02
        assert same_answers(a, b)
    # the mesh is reported as primitives Pb .. Pb + n - 1
    pb = len(base.flatten().prims)
    hit = np.concatenate([r[0] for r in a])
    assert ((hit > pb) & (hit <= pb + mesh.n_tris)).any()


def _whitted(ctx, camera):
    cam, fd = camera.pod(), camera.film.desc()
    film = np.zeros_like(camera.film.pixels)
    ctx.check(ctx.lib.trace_render_whitted(ctx.h, C.byref(cam), C.byref(fd), 2, 5, C.c_uint64(9), film.ctypes.data_as(C.c_void_p)))
    return film


def _sppm(T, ctx, camera):
    cam, fd = camera.pod(), camera.film.desc()
    h, w = camera.film.pixels.shape[:2]
    rgb = np.zeros((h, w, 3), np.float32)
    ctx.check(ctx.lib.trace_render_sppm(ctx.h, C.byref(cam), C.byref(fd), 0.3, 5, 3, 20_000, 0, C.c_uint64(3),
                                        C.cast(None, T._lib.SPPM_CB), None, rgb.ctypes.data_as(C.c_void_p)))
    return rgb


def test_images_match(T, dctx, hctx):
    for name in ("tess_small", "caustic"):
        base, mesh, camera = split_case(T, name, 1)
        cs = T.CompositeScene(base, mesh)
        dctx.upload(cs)
        upload_d(T, hctx, base, mesh)
        a, b = _whitted(dctx, camera), _whitted(hctx, camera)
        assert float(a[..., :3].max()) > 0 and same_image(a, b)
        if name == "caustic":
            a, b = _sppm(T, dctx, camera), _sppm(T, hctx, camera)
            assert float(a.max()) > 0 and same_image(a, b)
        # the integrator functors take the composite scene
        T.WhittedIntegrator(camera, T.UniformSampler(1), 5, context=dctx)(cs)
        assert float(camera.film.pixels[..., 3].max()) > 0
        assert float(T.SPPMIntegrator(camera, 0.3, 5, 1, 20_000, context=dctx)(cs).max()) > 0


def test_attach_sequence_keeps_the_base(T, dctx, hctx, sctx):
    base, _, camera = split_case(T, "tess_small", 1)
    nb = len(base.flatten().nodes)
    rays = ray_families(T, T.CompositeScene(base, sphere_mesh(T, (2.5, 2.0, -20.0), 2.0, 8, 10)), camera, 100_000, seed=3)
    first = None
    for stacks, slices in ((8, 10), (30, 40), (5, 6)):       # grow, then shrink
        mesh = sphere_mesh(T, (2.5, 2.0, -20.0), 2.0, stacks, slices)
        dctx.upload(T.CompositeScene(base, mesh))
        nodes, sh = dctx.scene_nodes(), dctx.shadow_tree()
        dn, _ = upload_d(T, hctx, base, mesh)
        assert same_bits(nodes, dn) and same_bits(nodes, hctx.scene_nodes())
        assert same_bits(sh, expected_shadow(sctx, base, mesh, int(dn[0]["meta"]) >> 30))
        assert same_answers(answers(dctx, rays), answers(hctx, rays))
        part = (nodes[1:1 + nb].tobytes(), sh[1:len(base.flatten().prims)].tobytes())
        first = first or part
        assert part == first                                   # the base's records are untouched by later attaches


def test_refit_after_attach_and_attach_after_refit(T, dctx, hctx, sctx):
    import torch
    base, mesh, camera = split_case(T, "tess_small", 1)
    flat = base.flatten()
    cs = T.CompositeScene(base, mesh)
    dctx.upload(cs)
    upload_d(T, hctx, base, mesh)
    mv = mesh.vertices.cpu().numpy()
    bv = wave(flat, 1.5, seed=3)
    moved = np.concatenate([bv, mv + np.float32(0.5)]).astype(np.float32)
    rays = ray_families(T, cs, camera, 200_000, seed=5)
    sctx.upload(base)                                          # (the base refit alone: the reference of the next attach)
    sctx.refit(base, bv)
    base_nodes = sctx.scene_nodes()
    dctx.refit(cs, torch.from_numpy(moved).cuda(0))
    hctx.check(hctx.lib.trace_scene_refit(hctx.h, len(moved), T._lib.ptr(moved), None, 0, None))
    assert same_bits(dctx.scene_nodes(), hctx.scene_nodes())
    assert same_answers(answers(dctx, rays), answers(hctx, rays))
    with pytest.raises(ValueError, match="vertices of all its triangles"):
        dctx.refit(cs)
    # the next attach composes with the refit base: D over the base refit alone
    mesh2 = sphere_mesh(T, (2.5, 3.0, -20.0), 1.5, 12, 14)
    dctx.upload(T.CompositeScene(base, mesh2))
    dn, _ = upload_d(T, hctx, base, mesh2, base_nodes=base_nodes, base_vertices=bv)
    assert same_bits(dctx.scene_nodes(), dn) and same_bits(dctx.scene_nodes(), hctx.scene_nodes())
    assert same_answers(answers(dctx, rays), answers(hctx, rays))


def _raw_attach(ctx, mesh, n_tris=None):
    d, keep = mesh.desc(ctx.device)
    if n_tris is not None:
        d.n_tris = n_tris
    return ctx.lib.trace_scene_attach_mesh_device(ctx.h, C.byref(d), None)


def test_refusals_keep_the_previous_scene(T, dctx):
    base, mesh, camera = split_case(T, "tess_small", 1)
    cs = T.CompositeScene(base, mesh)
    dctx.upload(cs)
    rays = ray_families(T, cs, camera, 50_000, seed=1)
    before, nodes, sh = answers(dctx, rays), dctx.scene_nodes(), dctx.shadow_tree()
    v = mesh.vertices.cpu().numpy()
    bad_v = v.copy()
    bad_v[7, 1, 2] = np.nan
    bad_n = np.ones_like(v)
    bad_n[3, 0, 0] = np.nan
    pts = deep_bounds()[:, :3]
    deep = np.repeat(pts[:, None, :], 3, axis=1).astype(np.float32)
    mat = mesh.materials
    cases = [(T.DeviceMeshScene([], _dev(bad_v), mat), "NaN in a triangle vertex"),
             (T.DeviceMeshScene([], _dev(v), mat, normals=_dev(bad_n)), "NaN in a triangle normal"),
             (T.DeviceMeshScene([], _dev(v), mat, _dev(np.full(len(v), 1, np.int32))), "material index is out of range"),
             (T.DeviceMeshScene([], _dev(deep), mat), "deeper than 64 levels")]
    for bad, msg in cases:
        with pytest.raises(RuntimeError, match=msg):
            dctx.upload(T.CompositeScene(base, bad))
        assert dctx._mesh is mesh
        assert same_bits(dctx.scene_nodes(), nodes) and same_bits(dctx.shadow_tree(), sh)
        assert same_answers(answers(dctx, rays), before)
    assert _raw_attach(dctx, mesh, n_tris=0) != 0 and b"n_tris must be in [1" in dctx.lib.trace_last_error(dctx.h)
    assert same_answers(answers(dctx, rays), before)
    fresh = T.Context(0)
    try:
        assert _raw_attach(fresh, mesh) != 0 and b"no scene uploaded" in fresh.lib.trace_last_error(fresh.h)
        fresh.upload(T.DeviceMeshScene([], np.zeros((0, 3, 3), np.float32), mat))
        assert _raw_attach(fresh, mesh) != 0 and b"has no primitive" in fresh.lib.trace_last_error(fresh.h)
    finally:
        fresh.close()


def _depth64_points():
    """point boxes (a subset of deep_bounds) whose radix tree with one primitive per leaf is exactly 64 levels deep"""
    b = deep_bounds()
    for k in range(len(b), 1, -1):
        if lbvh_restate(b[:k], 1)[2] == 64:
            return b[:k, :3]
    raise AssertionError("no subset of deep_bounds is 64 levels deep")


def test_depth_rule(T, dctx, hctx, sctx):
    pts = _depth64_points()
    m = T.MatteMaterial(T.ConstantTexture(T.RGBSpectrum(0.5)), T.ConstantTexture(0.0))
    core = T.ShapeCore(T.Transformation(), False)
    tris = [T.GeometricPrimitive(t, m) for p in pts for t in T.create_triangle_mesh(core, 1, [1, 2, 3], 3, [p, p, p])]
    base = T.Scene([], T.BVHAccel(tris, 4, builder="lbvh"))
    sctx.upload(base)
    st = sctx.shadow_tree()
    assert st is not None and len(st) == len(pts) - 1               # the base alone keeps its 64-level shadow tree
    mesh = sphere_mesh(T, (4.0, 4.0, 4.0), 1.0, 6, 8)
    cs = T.CompositeScene(base, mesh)
    dctx.upload(cs)
    assert dctx.shadow_tree() is None                               # 1 + 64 levels: no composed shadow tree
    upload_d(T, hctx, base, mesh)
    assert same_bits(dctx.scene_nodes(), hctx.scene_nodes())
    rng = np.random.default_rng(6)
    o = rng.uniform(-2, 10, (100_000, 3)).astype(np.float32)
    d = (np.float32(4.0) + rng.normal(size=(100_000, 3)).astype(np.float32) - o).astype(np.float32)
    rays = [(o, d, None), (o, d, rng.uniform(0.2, 1.2, 100_000).astype(np.float32))]
    a, b = answers(dctx, rays), answers(hctx, rays)
    assert (a[0][0] != 0).mean() > 0.01 and same_answers(a, b)


def test_deterministic_and_flat_memory(T, dctx):
    import torch
    base, _, _ = split_case(T, "tess_small", 1)
    out = []
    for _ in range(2):
        dctx.upload(T.CompositeScene(base, sphere_mesh(T, (2.5, 2.0, -20.0), 2.0, 20, 24)))
        out.append((dctx.scene_nodes(), dctx.shadow_tree()))
    assert same_bits(out[0][0], out[1][0]) and same_bits(out[0][1], out[1][1])
    mesh = sphere_mesh(T, (2.5, 2.0, -20.0), 2.0, 20, 24)
    mk = lambda: T.DeviceMeshScene([], mesh.vertices, mesh.materials, None, mesh.normals, mesh.flags)
    for _ in range(2):
        dctx.upload(T.CompositeScene(base, mk()))
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(0)[0]
    for _ in range(3):
        dctx.upload(T.CompositeScene(base, mk()))
    torch.cuda.synchronize()
    assert torch.cuda.mem_get_info(0)[0] == free0
