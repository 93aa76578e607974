"""Refit (trace_scene_refit, csrc/refit.cu) restated in numpy, checked without a GPU.  `refit_restate` is the
specification tests/test_gpu_refit.py holds the device to, bit for bit: over an uploaded flat's topology, a leaf's box
is the Julia-order min / max of its primitives' bounds (a triangle's vertices, a sphere's world bound), an interior
box the union of its children's, and a node whose subtree holds no primitive (a zero-primitive leaf, Q16) keeps its box
and adds nothing to its parent's."""
import copy

import numpy as np
import pytest

import oracle_lib
from test_gpu_lbvh import _jl_float, _jl_key


def refit_restate(flat, vertices=None):
    """-> nodes (node_dtype): flat.nodes with every box recomputed from `vertices` ([n_tris, 3, 3], default the flat's)"""
    from trace_jl_b200 import _lib as tl
    nodes = flat.nodes.copy()
    n = len(nodes)
    if n == 0:
        return nodes
    v = flat.tri_vertices if vertices is None else np.asarray(vertices, np.float32).reshape(-1, 3, 3)
    prims = flat.prims
    # primitive bounds as Julia-order keys; (0xFFFFFFFF, 0) is the empty box (no float has key 0xFFFFFFFF)
    pk = np.empty((len(prims), 6), np.uint32)
    tri = prims["kind"] == tl.PRIM_TRIANGLE
    if tri.any():
        tk = _jl_key(v[prims["index"][tri].astype(np.int64)])
        pk[tri, :3], pk[tri, 3:] = tk.min(1), tk.max(1)
    if (~tri).any():
        pk[~tri] = _jl_key(flat.sphere_bounds[prims["index"][~tri].astype(np.int64)])
    meta = nodes["meta"].astype(np.int64)
    off = nodes["offset"].astype(np.int64)
    leaf = (meta >> 30) == 3
    cnt = np.where(leaf, meta & 0x3FFFFFFF, 0)
    box = np.empty((n, 6), np.uint32)
    box[:, :3], box[:, 3:] = 0xFFFFFFFF, 0
    full = np.nonzero(cnt > 0)[0]
    full = full[np.argsort(off[full])]
    starts = off[full]
    assert np.array_equal(np.append(starts[1:], len(prims)), starts + cnt[full])    # the leaves tile the primitive list
    if len(full):
        box[full, :3] = np.minimum.reduceat(pk[:, :3], starts, axis=0)
        box[full, 3:] = np.maximum.reduceat(pk[:, 3:], starts, axis=0)
    # depth of every node (preorder: first child = parent + 1, second = offset), then unions from the deepest level up
    depth = np.zeros(n, np.int64)
    level = np.array([0])
    d = 0
    while len(level):
        depth[level] = d
        inner = level[~leaf[level]]
        level = np.concatenate([inner + 1, off[inner]])
        d += 1
    for lv in range(d - 1, -1, -1):
        i = np.nonzero((depth == lv) & ~leaf)[0]
        a, b = i + 1, off[i]
        box[i, :3] = np.minimum(box[a, :3], box[b, :3])
        box[i, 3:] = np.maximum(box[a, 3:], box[b, 3:])
    has = box[:, 0] != 0xFFFFFFFF
    nodes["bmin"][has] = _jl_float(box[has, :3])
    nodes["bmax"][has] = _jl_float(box[has, 3:])
    return nodes


def refit_flat(flat, vertices, normals=None):
    """A flat with the same topology, new vertices (and normals) and restated boxes: what a refit leaves on the device"""
    out = copy.copy(flat)
    out.tri_vertices = np.ascontiguousarray(vertices, np.float32).reshape(-1, 3, 3)
    if normals is not None:
        out.tri_normals = np.ascontiguousarray(normals, np.float32).reshape(-1, 3, 3)
    out.nodes = refit_restate(flat, out.tri_vertices)
    out.stale = False
    return out


def boxes_equal(a, b):
    """float == of the boxes (the sign of a zero may differ), structure words identical"""
    return (np.array_equal(a["bmin"], b["bmin"]) and np.array_equal(a["bmax"], b["bmax"]) and
            np.array_equal(a["offset"], b["offset"]) and np.array_equal(a["meta"], b["meta"]))


def wave(flat, amplitude, seed=0):
    """Heightfield-style deformation of every triangle vertex: y += A sin(1.3 x + phase) cos(0.9 z + phase')"""
    rng = np.random.default_rng(seed)
    ph = rng.uniform(0, 2 * np.pi, 2)
    v = flat.tri_vertices.astype(np.float64)
    v[..., 1] += amplitude * np.sin(1.3 * v[..., 0] + ph[0]) * np.cos(0.9 * v[..., 2] + ph[1])
    return v.astype(np.float32)


def tess_small(T, builder="reference", max_node_primitives=1):
    return T.scenes.tessellated(cells=48, stacks=26, slices=24, res=(160, 90), builder=builder,
                                max_node_primitives=max_node_primitives)


def nested_scene(T):
    """A mesh, loose triangles and spheres, with a BVHAccel of spheres and triangles nested as one primitive"""
    rng = np.random.default_rng(1)
    mk = lambda c, r: T.GeometricPrimitive(T.Sphere(T.ShapeCore(T.translate(c), False), r, 360.0))
    core = T.ShapeCore(T.Transformation(), False)
    v, _, idx = T.scenes._heightfield(6)
    mesh = T.TriangleSet(core, T.TriangleMesh(core.object_to_world, len(idx), idx.reshape(-1), len(v), v))
    loose = T.create_triangle_mesh(core, 2, [1, 2, 3, 2, 3, 4], 4, [(0, 0, -12), (1, 0, -12), (0, 1, -12), (1, 1, -12)])
    inner = [mk(rng.uniform(-4, 0, 3) + [0, 0, -20], 0.6) for _ in range(4)] + [T.GeometricPrimitive(t) for t in loose]
    outer = [mk(rng.uniform(0, 4, 3) + [0, 0, -20], 0.5) for _ in range(3)] + [T.PrimitiveBatch(mesh, None)]
    return T.Scene([], T.BVHAccel(outer + [T.BVHAccel(inner)]))


def scenes_for_identity(T):
    out = {"tess_reference": tess_small(T)[0], "tess_sah": tess_small(T, "sah")[0],
           "shadows": T.scenes.shadows(resolution=32)[0], "nested": nested_scene(T)}
    scene, _, _ = T.scenes.shadows(resolution=32)
    out["shadows_mixed_leaves"] = T.Scene(scene.lights, T.BVHAccel([p for _, p in scene.aggregate.items], 4))
    return out


@pytest.mark.parametrize("name", ["tess_reference", "tess_sah", "shadows", "shadows_mixed_leaves", "nested"])
def test_identity_restatement_reproduces_tree(T, name):
    flat = scenes_for_identity(T)[name].flatten()
    assert boxes_equal(refit_restate(flat), flat.nodes)
    if name == "shadows_mixed_leaves":
        meta = flat.nodes["meta"].astype(np.int64)
        kinds = [set(flat.prims["kind"][o:o + (m & 0x3FFFFFFF)].tolist())
                 for o, m in zip(flat.nodes["offset"].astype(np.int64), meta) if (m >> 30) == 3]
        assert any(len(k) == 2 for k in kinds)          # a leaf holding a sphere and a triangle


def test_identity_restatement_caustic_zero_primitive_leaves(T):
    import os
    if not os.path.exists(T.scenes.ASSET_PLY):
        pytest.skip("asset missing")
    flat = T.scenes.caustic_glass()[0].flatten()
    meta = flat.nodes["meta"].astype(np.int64)
    assert (((meta >> 30) == 3) & ((meta & 0x3FFFFFFF) == 0)).any()
    assert boxes_equal(refit_restate(flat), flat.nodes)


def test_restated_tree_gives_fresh_tree_hits(T):
    """The oracle walking the refit tree over deformed vertices finds the same t, bit for bit, as on a reference tree
    built for the deformed geometry (the primitive may differ on ties of equal t)."""
    scene, camera, _ = tess_small(T)
    flat = scene.flatten()
    new = wave(flat, 1.5, seed=3)
    # the same geometry as a fresh scene: move the meshes' vertices, build a new tree
    meshes = flat.tri_sources
    pos = 0
    for m in meshes:
        k = m.n_triangles
        idx = m.indices.reshape(-1, 3).astype(np.int64) - 1
        m.vertices[idx.reshape(-1)] = new[pos:pos + k].reshape(-1, 3)
        pos += k
    assert np.array_equal(flat.gather_vertices(), new)
    fresh = T.Scene(scene.lights, T.BVHAccel([p for _, p in scene.aggregate.items], 1)).flatten()
    rf = refit_flat(flat, new)
    assert not boxes_equal(rf.nodes, flat.nodes)
    rng = np.random.default_rng(5)
    lo, hi = fresh.nodes[0]["bmin"], fresh.nodes[0]["bmax"]
    n = 60_000
    tgt = (lo + rng.random((n, 3), dtype=np.float32) * (hi - lo)).astype(np.float32)
    o = (tgt + rng.normal(size=(n, 3)).astype(np.float32) * 8).astype(np.float32)
    d = (tgt - o).astype(np.float32)
    pa, ta, _ = oracle_lib.OracleScene(rf).intersect(o, d, slab=0)
    pb, tb, _ = oracle_lib.OracleScene(fresh).intersect(o, d, slab=0)
    assert (pa != 0).mean() > 0.3
    assert np.array_equal(ta.view(np.uint32), tb.view(np.uint32))
    assert (pa != pb).mean() < 1e-3


def test_gather_order_is_flattening_order(T):
    """Context.refit(scene) with vertices=None uploads FlatScene.gather_vertices(): the meshes' vertices in the order
    of tri_vertices, batches and single triangles (nested BVHAccels included) alike."""
    for scene in (nested_scene(T), T.scenes.shadows(resolution=32)[0], tess_small(T)[0]):
        flat = scene.flatten()
        assert np.array_equal(flat.gather_vertices(), flat.tri_vertices)
        assert len(flat.sphere_bounds) == len(flat.spheres)


def test_stale_flat_is_not_uploaded(T):
    """After a refit the host flat no longer describes the device scene: no context may upload it."""
    flat = T.scenes.shadows(resolution=32)[0].flatten()
    flat.stale = True
    ctx = object.__new__(T.Context)          # no device needed: the refusal comes before any library call
    ctx._scene = None
    scene = T.Scene([], T.BVHAccel([]))
    scene._flat = flat
    with pytest.raises(RuntimeError, match="stale"):
        ctx.upload(scene)
