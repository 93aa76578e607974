"""The device mesh upload (trace_scene_upload_mesh_device, csrc/upload_device.cu; DeviceMeshScene + Context.upload).
Its contract: the device scene is bit for bit the one trace_scene_upload builds from the LBVH of the triangles' Julia
min / max boxes and prims[k] = {TRIANGLE, order[k], material[order[k]], order[k]}.  Checked here against
`lbvh_restate`, against the host path (BVHAccel(builder="lbvh") + Context.upload) and against that exact host upload
made by hand in a second context; then images, refit, refusals, determinism and memory."""
import ctypes as C
import os

import numpy as np
import pytest

from test_gpu_lbvh import _jl_float, _jl_key, deep_bounds, gpu_build, lbvh_restate, same_bits
from test_gpu_parity import camera_rays
from test_gpu_refit import same_image
from test_refit_host import boxes_equal, tess_small, wave

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


def host_scene(T, name, m):
    """(scene, camera) of the host path, BVHAccel(builder="lbvh")"""
    if name == "tess_small":
        scene, camera, _ = tess_small(T, "lbvh", m)
    elif name == "tess_1M":
        scene, camera, _ = T.scenes.tessellated(res=(192, 108), builder="lbvh", max_node_primitives=m)
    else:
        if not os.path.exists(T.scenes.ASSET_PLY):
            pytest.skip("asset missing")
        scene, camera, _ = T.scenes.caustic_glass(resolution=64, builder="lbvh", max_node_primitives=m)
    return scene, camera


def mesh_arrays(flat):
    """the per-triangle arrays of a flattened triangle scene: vertices, normals, flags, material ids"""
    n = len(flat.tri_vertices)
    ids = np.zeros(n, np.uint32)
    ids[flat.prims["index"].astype(np.int64)] = flat.prims["material"]
    return flat.tri_vertices, flat.tri_normals, flat.tri_flags, ids


def device_scene(T, scene, m, **kw):
    import torch
    flat = scene.flatten()
    v, nrm, f, ids = mesh_arrays(flat)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda(0)
    return T.DeviceMeshScene(scene.lights, dev(v), flat.materials, dev(ids.astype(np.int32)), dev(nrm), dev(f),
                             max_node_primitives=m, **kw)


def jl_bounds(v):
    """Julia min / max of each triangle's three vertices, [n, 6]"""
    k = _jl_key(np.ascontiguousarray(v, np.float32))
    return np.concatenate([_jl_float(k.min(1)), _jl_float(k.max(1))], 1).astype(np.float32)


def contract_upload(T, ctx, scene, m):
    """trace_scene_upload of the contract's inputs, made by hand: -> number of nodes"""
    flat = scene.flatten()
    v, nrm, f, ids = mesh_arrays(flat)
    rc, nodes, order = gpu_build(jl_bounds(v), m)
    assert rc == 0
    prims = np.zeros(len(order), T._lib.prim_dtype)
    prims["kind"], prims["index"], prims["material"], prims["original"] = T._lib.PRIM_TRIANGLE, order, ids[order], order
    keep = [nodes, prims, v, nrm, f, flat.materials_pod, flat.lights]
    d = T._lib.SceneDesc()
    d.n_nodes, d.nodes = len(nodes), T._lib.ptr(nodes)
    d.n_prims, d.prims = len(prims), T._lib.ptr(prims)
    d.n_tris, d.tri_vertices, d.tri_normals, d.tri_flags = len(v), T._lib.ptr(v), T._lib.ptr(nrm), T._lib.ptr(f)
    d.n_spheres, d.spheres = 0, None
    d.n_materials, d.materials = flat.n_materials, T._lib.ptr(flat.materials_pod)
    d.n_lights, d.lights = len(flat.lights), T._lib.ptr(flat.lights)
    ctx.check(ctx.lib.trace_scene_upload(ctx.h, C.byref(d)))
    ctx._scene, ctx._n_nodes = object(), len(nodes)       # (a scene Context.upload did not make: never cached)
    del keep
    return len(nodes)


def ray_families(T, scene, camera, n, seed):
    """camera rays, and segments towards random points of the scene box (t_max 0.2 .. 1.2 of the segment)"""
    rng = np.random.default_rng(seed)
    o1, d1 = camera_rays(T, camera, n, rng)
    b = scene.bound
    tgt = (b.p_min + rng.random((n, 3), dtype=np.float32) * (b.p_max - b.p_min)).astype(np.float32)
    o2 = (tgt + rng.normal(size=(n, 3)).astype(np.float32) * np.float32(0.1 * float(np.max(b.p_max - b.p_min)))).astype(np.float32)
    d2 = (tgt - o2).astype(np.float32)
    t2 = rng.uniform(0.2, 1.2, n).astype(np.float32)
    return [(o1, d1, None), (o2, d2, t2)]


def answers(ctx, rays):
    out = []
    for o, d, t in rays:
        p, th, bc = ctx.intersect(o, d, t)
        out.append((p, th.view(np.uint32), bc.view(np.uint32), ctx.occluded(o, d, t)))
    return out


def same_answers(a, b):
    return all(np.array_equal(x, y) for ra, rb in zip(a, b) for x, y in zip(ra, rb))


@pytest.mark.parametrize("m", [1, 4])
@pytest.mark.parametrize("name", ["tess_small", "caustic", "tess_1M"])
def test_tree_and_exact_contract(T, dctx, hctx, name, m):
    scene, camera = host_scene(T, name, m)
    ds = device_scene(T, scene, m)
    assert dctx.upload(ds) is ds
    nodes = dctx.scene_nodes()
    # 1. the tree: the restatement bit for bit; the host path's with boxes float == (numpy may pick the other zero)
    rnodes, _, _ = lbvh_restate(jl_bounds(scene.flatten().tri_vertices), m)
    assert same_bits(nodes, rnodes)
    hctx.upload(scene)
    assert boxes_equal(nodes, hctx.scene_nodes())
    # 2. the exact contract: the host upload of the contract's inputs, made by hand
    n_nodes = contract_upload(T, hctx, scene, m)
    assert n_nodes == len(nodes) and same_bits(hctx.scene_nodes(), nodes)
    sd, sh = dctx.shadow_tree(), hctx.shadow_tree()
    assert sd is not None and same_bits(sd, sh)
    n = 1_000_000 if name != "tess_small" else 200_000
    rays = ray_families(T, scene, camera, n, seed=7 + m)
    a, b = answers(dctx, rays), answers(hctx, rays)
    assert (a[0][0] != 0).mean() > 0.02 and a[1][3].mean() > 0.02
    assert same_answers(a, b)


def _whitted(ctx, scene, camera):
    ctx.upload(scene)
    cam, fd = camera.pod(), camera.film.desc()
    film = np.zeros_like(camera.film.pixels)
    ctx.check(ctx.lib.trace_render_whitted(ctx.h, C.byref(cam), C.byref(fd), 2, 5, C.c_uint64(9), film.ctypes.data_as(C.c_void_p)))
    return film


def _sppm(T, ctx, scene, camera):
    ctx.upload(scene)
    cam, fd = camera.pod(), camera.film.desc()
    h, w = camera.film.pixels.shape[:2]
    rgb = np.zeros((h, w, 3), np.float32)
    ctx.check(ctx.lib.trace_render_sppm(ctx.h, C.byref(cam), C.byref(fd), 0.3, 5, 3, 20_000, 0, C.c_uint64(3),
                                        C.cast(None, T._lib.SPPM_CB), None, rgb.ctypes.data_as(C.c_void_p)))
    return rgb


def test_images_equal_host_path(T, dctx, hctx):
    scene, camera = host_scene(T, "tess_small", 1)
    ds = device_scene(T, scene, 1)
    a, b = _whitted(dctx, ds, camera), _whitted(hctx, scene, camera)
    assert float(a[..., :3].max()) > 0 and same_image(a, b)
    # the integrator functors take the scene unchanged
    T.WhittedIntegrator(camera, T.UniformSampler(1), 5, context=dctx)(ds)
    assert float(camera.film.pixels[..., 3].max()) > 0
    scene, camera = host_scene(T, "caustic", 1)
    ds = device_scene(T, scene, 1)
    a, b = _whitted(dctx, ds, camera), _whitted(hctx, scene, camera)
    assert float(a[..., :3].max()) > 0 and same_image(a, b)
    a, b = _sppm(T, dctx, ds, camera), _sppm(T, hctx, scene, camera)
    assert float(a.max()) > 0 and same_image(a, b)
    img = T.SPPMIntegrator(camera, 0.3, 5, 1, 20_000, context=dctx)(ds)
    assert float(img.max()) > 0


@pytest.mark.parametrize("m", [1, 4])
def test_refit_after_device_upload(T, dctx, hctx, m):
    import torch
    scene, camera = host_scene(T, "tess_small", m)
    flat = scene.flatten()
    new = wave(flat, 1.5, seed=3)
    ds = device_scene(T, scene, m)
    dctx.upload(ds)
    hctx.upload(scene)
    dctx.refit(ds, torch.from_numpy(new).cuda(0))
    hctx.refit(scene, new)
    nodes = dctx.scene_nodes()
    assert boxes_equal(nodes, hctx.scene_nodes()) and not boxes_equal(nodes, flat.nodes)
    rays = ray_families(T, scene, camera, 200_000, seed=5)
    assert same_answers(answers(dctx, rays), answers(hctx, rays))
    assert same_bits(dctx.shadow_tree(), hctx.shadow_tree())
    # the tensor-in-place form: the scene's own tensor, changed by the caller, equals passing the tensor
    ds2 = device_scene(T, scene, m)
    dctx.upload(ds2)
    ds2.vertices.copy_(torch.from_numpy(new))
    dctx.refit(ds2)
    assert same_bits(dctx.scene_nodes(), nodes)


def _good_scene(T):
    scene, camera = host_scene(T, "tess_small", 1)
    return scene, camera, device_scene(T, scene, 1)


def test_refusals_keep_the_previous_scene(T, dctx):
    import torch
    scene, camera, ds = _good_scene(T)
    dctx.upload(ds)
    rays = ray_families(T, scene, camera, 50_000, seed=1)
    before, nodes = answers(dctx, rays), dctx.scene_nodes()
    flat = scene.flatten()
    v, nrm, f, ids = mesh_arrays(flat)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda(0)
    bad_v, bad_n, bad_ids = v.copy(), nrm.copy(), ids.astype(np.int32)
    bad_v[123, 1, 2] = np.nan
    bad_n[77, 0, 0] = np.nan
    bad_ids[5] = len(flat.materials)
    pts = deep_bounds()[:, :3]
    deep = np.repeat(pts[:, None, :], 3, axis=1).astype(np.float32)
    cases = [(dict(vertices=dev(bad_v), normals=dev(nrm), flags=dev(f)), "NaN in a triangle vertex"),
             (dict(vertices=dev(v), normals=dev(bad_n), flags=dev(f)), "NaN in a triangle normal"),
             (dict(vertices=dev(v), material_ids=dev(bad_ids)), "material index is out of range"),
             (dict(vertices=dev(deep)), "deeper than 64 levels"),
             (dict(vertices=dev(deep), max_node_primitives=4), "deeper than 64 levels")]
    for kw, msg in cases:
        kw.setdefault("material_ids", None)
        bad = T.DeviceMeshScene(scene.lights, materials=flat.materials, **kw)
        with pytest.raises(RuntimeError, match=msg):
            dctx.upload(bad)
        assert dctx._scene is ds
        assert same_bits(dctx.scene_nodes(), nodes) and same_answers(answers(dctx, rays), before)
    # Python refuses what the library cannot check: CPU tensors, wrong dtype, non-contiguous, another device
    vt = dev(v)
    for kw, msg in [(dict(vertices=torch.from_numpy(v)), "CPU tensor"),
                    (dict(vertices=vt.double()), "dtype float32"),
                    (dict(vertices=vt.transpose(1, 2)), "contiguous"),
                    (dict(vertices=vt, flags=dev(f).int()), "dtype uint8"),
                    (dict(vertices=vt, material_ids=dev(ids.astype(np.float32))), "dtype int32")]:
        with pytest.raises(ValueError, match=msg):
            T.DeviceMeshScene(scene.lights, materials=flat.materials, **kw)
    with pytest.raises(ValueError, match="on device 0, the context is on device 1"):
        ds.desc(1)
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError, match="different devices"):
            T.DeviceMeshScene(scene.lights, vt, flat.materials, normals=dev(nrm).cuda(1))
    assert same_answers(answers(dctx, rays), before)


def test_deterministic_and_no_allocation_when_warm(T, dctx):
    import torch
    scene, camera, ds = _good_scene(T)
    out = []
    for _ in range(2):
        ds = device_scene(T, scene, 1)
        dctx.upload(ds)
        out.append((dctx.scene_nodes(), dctx.shadow_tree()))
    assert same_bits(out[0][0], out[1][0]) and same_bits(out[0][1], out[1][1])
    v = ds.vertices
    mk = lambda: T.DeviceMeshScene(scene.lights, v, ds.materials, ds.material_ids, ds.normals, ds.flags)
    for _ in range(2):
        dctx.upload(mk())
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(0)[0]
    for _ in range(3):
        dctx.upload(mk())
    torch.cuda.synchronize()
    assert torch.cuda.mem_get_info(0)[0] == free0


def test_zero_and_one_triangle(T, dctx, hctx):
    import torch
    m = T.MatteMaterial(T.ConstantTexture(T.RGBSpectrum(0.5)), T.ConstantTexture(0.0))
    ds = T.DeviceMeshScene([], np.zeros((0, 3, 3), np.float32), [m])
    dctx.upload(ds)
    assert len(dctx.scene_nodes()) == 0 and dctx.shadow_tree() is None
    o = np.zeros((64, 3), np.float32)
    d = np.tile(np.array([[0, 0, -1]], np.float32), (64, 1))
    p, t, _ = dctx.intersect(o, d)
    assert (p == 0).all() and not dctx.occluded(o, d).any()
    tri = np.array([[[-1, -1, -3], [1, -1, -3], [0, 1, -3]]], np.float32)
    core = T.ShapeCore(T.Transformation(), False)
    hs = T.Scene([], T.BVHAccel([T.GeometricPrimitive(t, m) for t in T.create_triangle_mesh(core, 1, [1, 2, 3], 3, tri[0])],
                                1, builder="lbvh"))
    ds = T.DeviceMeshScene([], torch.from_numpy(tri).cuda(0), [m])
    dctx.upload(ds)
    hctx.upload(hs)
    assert boxes_equal(dctx.scene_nodes(), hctx.scene_nodes()) and len(dctx.scene_nodes()) == 1
    rng = np.random.default_rng(2)
    d = (rng.uniform(-0.5, 0.5, (4096, 3)) + np.array([0, 0, -3])).astype(np.float32)
    o = np.zeros_like(d)
    a, b = dctx.intersect(o, d), hctx.intersect(o, d)
    assert (a[0] != 0).mean() > 0.2 and all(np.array_equal(x, y) for x, y in zip(a, b))
    assert np.array_equal(dctx.occluded(o, d), hctx.occluded(o, d))
