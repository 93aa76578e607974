"""Several attached meshes (trace_scene_attach_meshes_device, csrc/upload_device.cu; CompositeScene + Context.upload).
Its contract: after every call the device scene is bit for bit the scene trace_scene_upload builds from D = C(base,
G(0, k)) (tests/test_attach_meshes_host.py, `compose_meshes`), and its shadow tree is the recursive composition of the
parts' own.  Checked here against D uploaded by hand in a second context: nodes, shadow tree, ray answers under both
walks and with the shadow-tree walks on and off, images; then sequences of calls that replace, append, keep and drop
slots, refit, refusals, the shadow tree's depth rule, determinism and memory."""
import ctypes as C

import numpy as np
import pytest

from test_attach_meshes_host import Part, compose_meshes, mesh_part
from test_gpu_attach_mesh import _depth64_points, _dev, _host, _sppm, _whitted, split_case, sphere_mesh
from test_gpu_device_upload import answers, jl_bounds, ray_families, same_answers
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


def uv_mesh(T, center, radius, stacks, slices, m=1, normals=True, flags=True, n_materials=1):
    """a UV sphere of 2 slices (stacks - 1) triangles; without normals / flags on request, and with n_materials > 1
    material ids cycling through them"""
    v, n, idx = T.scenes._uv_sphere(center, radius, stacks, slices)
    i = idx.astype(np.int64).reshape(-1, 3) - 1
    mats = [T.MirrorMaterial(T.ConstantTexture(T.RGBSpectrum(0.9)))] + \
        [T.MatteMaterial(T.ConstantTexture(T.RGBSpectrum(0.2 + 0.1 * j)), T.ConstantTexture(0.0)) for j in range(n_materials - 1)]
    ids = _dev((np.arange(len(i)) % n_materials).astype(np.int32)) if n_materials > 1 else None
    return T.DeviceMeshScene([], _dev(v[i]), mats, ids, _dev(n[i]) if normals else None,
                             _dev(np.full(len(i), 2 if normals else 1, np.uint8)) if flags else None, max_node_primitives=m)


def few_tris(T, center, count, m=1):
    """1 or 2 triangles near `center`, without normals or flags"""
    c = np.asarray(center, np.float32)
    quad = np.array([[0, 0, 0], [0.4, 0, 0], [0.4, 0.4, 0.1], [0, 0.4, 0.1]], np.float32) + c
    tri = np.stack([quad[[0, 1, 2]], quad[[0, 2, 3]]])[:count]
    mat = T.MatteMaterial(T.ConstantTexture(T.RGBSpectrum(0.7)), T.ConstantTexture(0.0))
    return T.DeviceMeshScene([], _dev(tri), [mat], max_node_primitives=m)


def _mesh_arrays(mesh, vertices=None):
    mv = _host(mesh.vertices) if vertices is None else vertices
    n = len(mv)
    mn = _host(mesh.normals)
    mf = np.zeros(n, np.uint8) if mesh.flags is None else _host(mesh.flags)
    if mn is None:
        mn, mf = np.zeros_like(mv), mf & ~np.uint8(2)
    mids = np.zeros(n, np.uint32) if mesh.material_ids is None else _host(mesh.material_ids).astype(np.uint32)
    return mv, mn, mf, mids


def _shadow_levels(pairs):
    u = pairs.view(np.uint32)
    best, stack = 0, [(0, 1)]
    while stack:
        i, d = stack.pop()
        best = max(best, d + 1)
        stack += [(int(u[i, c]), d + 1) for c in (6, 14) if not u[i, c] & 0x80000000]
    return best


def _part_shadow(sctx, scene, n_prims, single_box):
    """(pairs, single box, levels) of a part's own shadow tree, uploaded alone in sctx (levels 0: it has none)"""
    sctx.upload(scene)
    if n_prims == 1:
        return None, single_box, 1
    sh = sctx.shadow_tree()
    return (sh, None, _shadow_levels(sh)) if sh is not None else (None, None, 0)


def expected(T, sctx, base, meshes, base_state=None, mesh_state=None):
    """D as a Part (nodes, prims, shadow tree) and its arrays.  base_state / mesh_state[j]: (nodes, vertices, shadow
    pairs) of the base / mesh j after a refit, each refit alone; default: as uploaded"""
    flat = base.flatten()
    if base_state is None:
        bn, bv = flat.nodes, flat.tri_vertices
        bsh = _part_shadow(sctx, base, len(flat.prims), None)
    else:
        bn, bv, sh = base_state
        bsh = (sh, None, _shadow_levels(sh)) if sh is not None else (None, None, 0)
    bpart = Part(bn, flat.prims, len(flat.tri_vertices), flat.n_materials, *bsh)
    parts, arrays = [], []
    for j, mesh in enumerate(meshes):
        st = (mesh_state or {}).get(j)
        mv, mn, mf, mids = _mesh_arrays(mesh, None if st is None else st[1])
        rc, mnodes, morder = gpu_build(jl_bounds(_host(mesh.vertices)), mesh.max_node_primitives)
        assert rc == 0
        if st is None:
            b = jl_bounds(mv)
            msh = _part_shadow(sctx, mesh, len(mv), (b[0, :3], b[0, 3:]))
        else:
            mnodes = st[0]
            msh = (st[2], None, _shadow_levels(st[2])) if len(mv) > 1 else (None, (jl_bounds(mv)[0, :3], jl_bounds(mv)[0, 3:]), 1)
        parts.append(mesh_part(mnodes, morder, mids, len(mesh.materials), *msh))
        arrays.append((mv, mn, mf, mesh))
    d = compose_meshes(bpart, parts)
    v = np.concatenate([bv] + [a[0] for a in arrays]).astype(np.float32)
    nrm = np.concatenate([flat.tri_normals] + [a[1] for a in arrays]).astype(np.float32)
    f = np.concatenate([flat.tri_flags] + [a[2] for a in arrays]).astype(np.uint8)
    mats = [flat.materials_pod[:flat.n_materials]] + [a[3].desc(0)[1][0][:len(a[3].materials)] for a in arrays]
    lights = [flat.lights] + [a[3].desc(0)[1][1] for a in arrays]
    return d, (v, nrm, f, np.concatenate(mats), np.concatenate(lights), flat)


def upload_dk(T, ctx, d, arrays):
    """trace_scene_upload of D made by hand"""
    v, nrm, f, mats, lights, flat = arrays
    nodes, prims = np.ascontiguousarray(d.nodes), np.ascontiguousarray(d.prims)
    v, nrm, f = np.ascontiguousarray(v), np.ascontiguousarray(nrm), np.ascontiguousarray(f)
    mats, lights = np.ascontiguousarray(mats), np.ascontiguousarray(lights)
    sd = T._lib.SceneDesc()
    sd.n_nodes, sd.nodes = len(nodes), T._lib.ptr(nodes)
    sd.n_prims, sd.prims = len(prims), T._lib.ptr(prims)
    sd.n_tris, sd.tri_vertices, sd.tri_normals, sd.tri_flags = len(v), T._lib.ptr(v), T._lib.ptr(nrm), T._lib.ptr(f)
    sd.n_spheres, sd.spheres = len(flat.spheres), T._lib.ptr(flat.spheres)
    sd.n_materials, sd.materials = len(mats), T._lib.ptr(mats)
    sd.n_lights, sd.lights = len(lights), T._lib.ptr(lights)
    ctx.check(ctx.lib.trace_scene_upload(ctx.h, C.byref(sd)))
    ctx._scene, ctx._n_nodes, ctx._base, ctx._meshes = object(), len(nodes), None, []   # (never cached)


def check_d(T, dctx, hctx, sctx, base, meshes, rays=None, **state):
    """the device scene of dctx against D: nodes, shadow tree, and (rays) answers against D uploaded in hctx;
    -> (D, its arrays)"""
    d, arrays = expected(T, sctx, base, meshes, **state)
    nodes = dctx.scene_nodes()
    assert same_bits(nodes, d.nodes)
    sh = dctx.shadow_tree()
    assert (sh is None) == (d.shadow is None) and (sh is None or same_bits(sh, d.shadow))
    if rays is not None:
        upload_dk(T, hctx, d, arrays)
        assert same_bits(hctx.scene_nodes(), nodes)
        assert same_answers(answers(dctx, rays), answers(hctx, rays))
    return d, arrays


def all_ways(ctxs, rays):
    """answers under both walks, then with the shadow-tree walks off"""
    out = []
    for walk, tree in ((0, 1), (1, 1), (1, 0)):
        for c in ctxs:
            c.set_option("walk", walk)
            c.set_option("hit_tree", tree)
            c.set_option("shadow_tree", tree)
        out.append([answers(c, rays) for c in ctxs])
    for c in ctxs:
        c.set_option("walk", 1)
        c.set_option("hit_tree", 1)
        c.set_option("shadow_tree", 1)
    return out


def mesh_set(T, name, k, m):
    """k meshes around the base's region: 1, 2, ~1 k and 100 k triangles, with and without normals, flags and ids"""
    if name == "shadows":
        c, r = np.array([0.5, 0.6, -2.5]), 0.12
    elif name == "caustic":
        c, r = np.array([0.0, 1.0, -95.0]), 1.2
    else:
        c, r = np.array([2.5, 2.0, -20.0]), 1.5
    out = []
    for j in range(k):
        at = tuple(c + np.array([(j % 4 - 1.5) * 2.5 * r, (j // 4) * 2.5 * r, 0.0]))
        kind = j % 4
        if kind == 0:
            out.append(uv_mesh(T, at, r, 21, 26, m, n_materials=2))                       # 1040, normals, ids
        elif kind == 1:
            out.append(few_tris(T, at, 1 + (j // 4) % 2, m))                             # 1 or 2, bare
        elif kind == 2:
            out.append(uv_mesh(T, at, r, 251, 200, m, normals=False, flags=(j == 2)))     # 100 k
        else:
            out.append(uv_mesh(T, at, r, 12, 14, m, normals=True, flags=True, n_materials=3))
    return out


CASES = [("tess_small", 2, 1), ("caustic", 3, 4), ("tess_1M", 5, 1), ("shadows", 8, 4), ("tess_small", 8, 1)]


@pytest.mark.parametrize("name, k, m", CASES)
def test_exact_contract(T, dctx, hctx, sctx, name, k, m):
    base, _, camera = split_case(T, name, m)
    meshes = mesh_set(T, name, k, m)
    cs = T.CompositeScene(base, meshes)
    assert dctx.upload(cs) is cs
    d, arrays = check_d(T, dctx, hctx, sctx, base, meshes)
    assert (d.shadow is None) == (name == "shadows")
    upload_dk(T, hctx, d, arrays)
    assert same_bits(hctx.scene_nodes(), dctx.scene_nodes())
    rays = ray_families(T, cs, camera, 1_000_000, seed=17 + k)
    for a, b in all_ways([dctx, hctx], rays):
        assert same_answers(a, b)
    # the meshes are hit, reported as primitives after the base's
    hit = np.concatenate([r[0] for r in a])
    pb = len(base.flatten().prims)
    assert (hit > pb).any() and hit.max() <= pb + sum(m.n_tris for m in meshes)


def _raw(ctx, meshes):
    """trace_scene_attach_meshes_device with None as NULL, past Context.upload's cache: -> (rc, error text)"""
    descs = [None if m is None else m.desc(ctx.device) for m in meshes]
    arr = (ctx.lib.trace_scene_attach_meshes_device.argtypes[2]._type_ * max(1, len(meshes)))(
        *[C.pointer(x[0]) if x else None for x in descs])
    n_nodes = C.c_int64()
    rc = ctx.lib.trace_scene_attach_meshes_device(ctx.h, len(meshes), arr, C.byref(n_nodes))
    if rc == 0:
        ctx._n_nodes = n_nodes.value                           # (scene_nodes reads this many)
    return rc, ctx.lib.trace_last_error(ctx.h).decode() if rc else ""


def test_sequences(T, dctx, hctx, sctx):
    base, _, camera = split_case(T, "tess_small", 1)
    sph = lambda x, st, sl: sphere_mesh(T, (x, 2.0, -20.0), 1.0, st, sl)
    a, b, c = sph(0.0, 8, 10), sph(2.5, 10, 12), sph(5.0, 6, 8)
    rays = ray_families(T, T.CompositeScene(base, [a, b, c]), camera, 100_000, seed=4)
    steps = [[a, b, c], [a, sph(2.5, 30, 40), c], [a, sph(2.5, 5, 6), c]]        # the middle slot grows, then shrinks
    steps.append(steps[-1] + [sph(7.5, 9, 9)])                                   # append
    for meshes in steps:
        dctx.upload(T.CompositeScene(base, meshes))
        check_d(T, dctx, hctx, sctx, base, meshes, rays)
    before = dctx.scene_nodes()
    assert _raw(dctx, [None] * 4) == (0, "")                                    # keep all
    assert same_bits(dctx.scene_nodes(), before)
    check_d(T, dctx, hctx, sctx, base, steps[-1], rays)
    assert _raw(dctx, [None]) == (0, "")                                        # shrink to 1
    check_d(T, dctx, hctx, sctx, base, steps[-1][:1], rays)
    dctx._meshes = steps[-1][:1]
    dctx.upload(base)                                                            # a new upload clears the slots
    rc, err = _raw(dctx, [None])
    assert rc != 0 and "holds no mesh" in err
    # one call that replaces slots 0 and 2 equals the two replacements made one at a time
    x, y = sph(0.0, 14, 15), sph(5.0, 20, 9)
    dctx.upload(T.CompositeScene(base, [a, b, c, steps[-1][3]]))
    hctx.upload(T.CompositeScene(base, [a, b, c, steps[-1][3]]))
    dctx.upload(T.CompositeScene(base, [x, b, y, steps[-1][3]]))
    hctx.upload(T.CompositeScene(base, [x, b, c, steps[-1][3]]))
    hctx.upload(T.CompositeScene(base, [x, b, y, steps[-1][3]]))
    assert same_bits(dctx.scene_nodes(), hctx.scene_nodes()) and same_bits(dctx.shadow_tree(), hctx.shadow_tree())
    assert same_answers(answers(dctx, rays), answers(hctx, rays))
    check_d(T, dctx, hctx, sctx, base, [x, b, y, steps[-1][3]])
    # n_meshes = 1 equals trace_scene_attach_mesh_device
    dctx.upload(base)
    hctx.upload(base)
    assert _raw(dctx, [x]) == (0, "")
    d, keep = x.desc(0)
    n_nodes = C.c_int64()
    hctx.check(hctx.lib.trace_scene_attach_mesh_device(hctx.h, C.byref(d), C.byref(n_nodes)))
    hctx._n_nodes = n_nodes.value
    assert same_bits(dctx.scene_nodes(), hctx.scene_nodes()) and same_bits(dctx.shadow_tree(), hctx.shadow_tree())


def test_refit_then_keep(T, dctx, hctx, sctx):
    import torch
    base, _, camera = split_case(T, "tess_small", 1)
    flat = base.flatten()
    sph = lambda x, st, sl: sphere_mesh(T, (x, 2.0, -20.0), 1.0, st, sl)
    meshes = [sph(0.0, 8, 10), sph(2.5, 10, 12), sph(5.0, 6, 8)]
    cs = T.CompositeScene(base, meshes)
    dctx.upload(cs)
    d, arrays = expected(T, sctx, base, meshes)
    upload_dk(T, hctx, d, arrays)
    bv = wave(flat, 1.5, seed=3)
    mv = [_host(m.vertices) + np.float32(0.25 * (j + 1)) for j, m in enumerate(meshes)]
    moved = np.concatenate([bv] + mv).astype(np.float32)
    rays = ray_families(T, cs, camera, 200_000, seed=5)
    sctx.upload(base)                                          # (the base refit alone, before its flattening is stale)
    sctx.refit(base, bv)
    base_state = (sctx.scene_nodes(), bv, sctx.shadow_tree())
    dctx.refit(cs, torch.from_numpy(moved).cuda(0))
    hctx.check(hctx.lib.trace_scene_refit(hctx.h, len(moved), T._lib.ptr(moved), None, 0, None))
    assert same_bits(dctx.scene_nodes(), hctx.scene_nodes())
    assert same_answers(answers(dctx, rays), answers(hctx, rays))
    refit_shadow = dctx.shadow_tree()
    assert refit_shadow is not None
    # each part refit alone: its nodes and shadow tree as the device now holds them in the composed scene
    state = {}
    for j in (1, 2):
        sctx.upload(meshes[j])
        sctx.refit(meshes[j], torch.from_numpy(mv[j]).cuda(0))
        state[j] = (sctx.scene_nodes(), mv[j], sctx.shadow_tree())
    # keep all (only the top tree is written again), then replace slot 0 with a larger mesh: slots 1 and 2 move
    assert _raw(dctx, [None] * 3) == (0, "")
    assert same_bits(dctx.scene_nodes(), hctx.scene_nodes()) and same_bits(dctx.shadow_tree(), refit_shadow)
    new0 = sph(0.0, 30, 40)
    assert _raw(dctx, [new0, None, None]) == (0, "")
    d, arrays = check_d(T, dctx, hctx, sctx, base, [new0] + meshes[1:], base_state=base_state, mesh_state=state)
    upload_dk(T, hctx, d, arrays)
    assert same_answers(answers(dctx, rays), answers(hctx, rays))


def test_refusals_keep_the_previous_scene(T, dctx):
    base, _, camera = split_case(T, "tess_small", 1)
    sph = lambda x, st, sl: sphere_mesh(T, (x, 2.0, -20.0), 1.0, st, sl)
    meshes = [sph(0.0, 8, 10), sph(2.5, 10, 12), sph(5.0, 6, 8)]
    cs = T.CompositeScene(base, meshes)
    dctx.upload(cs)
    rays = ray_families(T, cs, camera, 50_000, seed=1)
    before, nodes, sh = answers(dctx, rays), dctx.scene_nodes(), dctx.shadow_tree()

    def unchanged():
        assert dctx._meshes == meshes
        assert same_bits(dctx.scene_nodes(), nodes) and same_bits(dctx.shadow_tree(), sh)
        assert same_answers(answers(dctx, rays), before)

    v = _host(meshes[2].vertices)
    bad_v = v.copy()
    bad_v[5, 2, 1] = np.nan
    mat = meshes[0].materials
    with pytest.raises(RuntimeError, match=r"NaN in a triangle vertex \(mesh 2"):
        dctx.upload(T.CompositeScene(base, [sph(0.0, 9, 9), sph(2.5, 7, 7), T.DeviceMeshScene([], _dev(bad_v), mat)]))
    unchanged()
    with pytest.raises(RuntimeError, match=r"material index is out of range \(mesh 1"):
        dctx.upload(T.CompositeScene(base, [meshes[0], T.DeviceMeshScene([], _dev(v), mat, _dev(np.full(len(v), 1, np.int32))), meshes[2]]))
    unchanged()
    for arg, msg in (([None] * 4, "slot 3 holds no mesh"), ([], "n_meshes must be in [1, 64], got 0"),
                     ([None] * 65, "n_meshes must be in [1, 64], got 65")):
        rc, err = _raw(dctx, arg)
        assert rc != 0 and msg in err
        unchanged()
    pts = _depth64_points()
    deep = T.DeviceMeshScene([], _dev(np.repeat(pts[:, None, :], 3, axis=1).astype(np.float32)), mat)
    with pytest.raises(RuntimeError, match=r"tree of mesh 1 is deeper than 63 levels"):
        dctx.upload(T.CompositeScene(base, [meshes[0], deep]))
    unchanged()
    ok = [meshes[0], sph(2.5, 11, 13), meshes[2]]
    dctx.upload(T.CompositeScene(base, ok))
    assert dctx._meshes == ok and not same_bits(dctx.scene_nodes(), nodes)


def test_shadow_tree_option_between_calls(T, dctx, hctx, sctx):
    """a kept mesh that moves while the option shadow_tree is off loses its shadow tree: no later call composes one
    from pairs left behind, and answers stay D's"""
    base, _, camera = split_case(T, "tess_small", 1)
    sph = lambda x, st, sl: sphere_mesh(T, (x, 2.0, -20.0), 1.0, st, sl)
    a, b, c = sph(0.0, 8, 10), sph(2.5, 10, 12), sph(5.0, 6, 8)
    rays = ray_families(T, T.CompositeScene(base, [a, b, c]), camera, 200_000, seed=8)

    def check(meshes, has_shadow):
        d, arrays = expected(T, sctx, base, meshes)
        assert same_bits(dctx.scene_nodes(), d.nodes)
        sh = dctx.shadow_tree()
        assert (sh is not None) == has_shadow
        if has_shadow:
            assert same_bits(sh, d.shadow)
        upload_dk(T, hctx, d, arrays)
        assert same_answers(answers(dctx, rays), answers(hctx, rays))

    try:
        dctx.upload(T.CompositeScene(base, [a, b, c]))
        check([a, b, c], True)
        dctx.set_option("shadow_tree", 0)
        big = sph(0.0, 30, 40)
        dctx.upload(T.CompositeScene(base, [big, b, c]))           # b and c move without their shadow pairs
        dctx.set_option("shadow_tree", 1)
        check([big, b, c], False)
        dctx.upload(T.CompositeScene(base, [sph(0.0, 30, 40), b, c]))   # same size: b and c stay where they are
        check([dctx._meshes[0], b, c], False)
        b2, c2 = sph(2.5, 10, 12), sph(5.0, 6, 8)
        dctx.upload(T.CompositeScene(base, [dctx._meshes[0], b2, c2]))  # rebuilt: a shadow tree again
        check([dctx._meshes[0], b2, c2], True)
        dctx.set_option("shadow_tree", 0)
        dctx.upload(T.CompositeScene(base, [sph(0.0, 5, 6), b2, c2]))    # moved down while off, then on: no stale read
        dctx.set_option("shadow_tree", 1)
        dctx.upload(T.CompositeScene(base, [sph(0.0, 4, 6), b2, c2]))
        check([dctx._meshes[0], b2, c2], False)
    finally:
        dctx.set_option("shadow_tree", 1)


def test_kept_mesh_too_deep_for_more_slots(T, dctx):
    base, _, camera = split_case(T, "tess_small", 1)
    small = sphere_mesh(T, (2.5, 2.0, -20.0), 1.0, 6, 8)
    pts = _depth64_points()
    deep = T.DeviceMeshScene([], _dev(np.repeat(pts[:, None, :], 3, axis=1).astype(np.float32)), small.materials)
    cs = T.CompositeScene(base, deep)
    dctx.upload(cs)                                             # 64 levels fit under a single slot
    rays = ray_families(T, cs, camera, 50_000, seed=2)
    before, nodes = answers(dctx, rays), dctx.scene_nodes()
    with pytest.raises(RuntimeError, match=r"tree of mesh 0 \(kept\) is deeper than 63 levels"):
        dctx.upload(T.CompositeScene(base, [deep, small]))      # the kept mesh would sit one level lower
    assert dctx._meshes == [deep] and same_bits(dctx.scene_nodes(), nodes)
    assert same_answers(answers(dctx, rays), before)
    rc, err = _raw(dctx, [None, small])
    assert rc != 0 and "(kept) is deeper than 63 levels" in err
    dctx.upload(T.CompositeScene(base, [small, small]))          # a new slot 0 is fine
    assert dctx._meshes == [small, small]


def _points_of_depth(levels):
    b = deep_bounds()
    for k in range(len(b), 1, -1):
        if lbvh_restate(b[:k], 1)[2] == levels:
            return b[:k, :3]
    raise AssertionError(f"no subset of deep_bounds is {levels} levels deep")


def test_depth_rule(T, dctx, hctx, sctx):
    base, _, camera = split_case(T, "tess_small", 1)
    small = sphere_mesh(T, (2.5, 2.0, -20.0), 1.0, 6, 8)
    mat = small.materials
    for levels, has in ((63, False), (62, True)):
        pts = _points_of_depth(levels)
        deep = T.DeviceMeshScene([], _dev(np.repeat(pts[:, None, :], 3, axis=1).astype(np.float32)), mat)
        dctx.upload(T.CompositeScene(base, [deep, small]))        # group: 1 + levels, D: 2 + levels
        assert (dctx.shadow_tree() is not None) == has
        d, _ = check_d(T, dctx, hctx, sctx, base, [deep, small])
        assert (d.shadow is not None) == has


def test_images_match(T, dctx, hctx, sctx):
    for name, k in (("tess_small", 3), ("caustic", 2)):
        base, _, camera = split_case(T, name, 1)
        meshes = mesh_set(T, name, k, 1)
        cs = T.CompositeScene(base, meshes)
        dctx.upload(cs)
        d, arrays = expected(T, sctx, base, meshes)
        upload_dk(T, hctx, d, arrays)
        a, b = _whitted(dctx, camera), _whitted(hctx, camera)
        assert float(a[..., :3].max()) > 0 and same_image(a, b)
        a, b = _sppm(T, dctx, camera), _sppm(T, hctx, camera)
        assert float(a.max()) > 0 and same_image(a, b)
        T.WhittedIntegrator(camera, T.UniformSampler(1), 5, context=dctx)(cs)
        assert float(camera.film.pixels[..., 3].max()) > 0


def test_deterministic_and_flat_memory(T, dctx):
    import torch
    base, _, _ = split_case(T, "tess_small", 1)
    src = [sphere_mesh(T, (x, 2.0, -20.0), 1.0, 20, 24) for x in (0.0, 2.5, 5.0)]
    mk = lambda m: T.DeviceMeshScene([], m.vertices, m.materials, None, m.normals, m.flags)
    out = []
    for _ in range(2):
        dctx.upload(base)
        dctx.upload(T.CompositeScene(base, [mk(m) for m in src]))
        out.append((dctx.scene_nodes(), dctx.shadow_tree()))
    assert same_bits(out[0][0], out[1][0]) and same_bits(out[0][1], out[1][1])
    meshes = [mk(m) for m in src]
    for j in range(3):                                               # replace each slot once (warm-up)
        meshes[j] = mk(src[j])
        dctx.upload(T.CompositeScene(base, list(meshes)))
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(0)[0]
    for rep in range(6):
        meshes[rep % 3] = mk(src[rep % 3])
        dctx.upload(T.CompositeScene(base, list(meshes)))
    torch.cuda.synchronize()
    assert torch.cuda.mem_get_info(0)[0] == free0
    assert same_bits(dctx.scene_nodes(), out[0][0]) and same_bits(dctx.shadow_tree(), out[0][1])
