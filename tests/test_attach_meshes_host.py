"""Several attached meshes, host side, without a GPU (trace_scene_attach_meshes_device, csrc/upload_device.cu;
CompositeScene + Context.upload).  `compose_parts` is the two-part composition C of the header, `compose_meshes`
applies it recursively: D = C(base, G(0, k)) with its shadow tree.  tests/test_gpu_attach_meshes.py holds the device to
it bit for bit, so it is checked here against the single-mesh restatement (`compose_restate` / `compose_shadow`) at
k = 1 and for its invariants on trees made by hand.  Also: the ctypes binding against the header, CompositeScene's
argument checks and the per-slot caching of Context.upload with the library call stubbed."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from test_attach_mesh_host import (REF_LEAF, REF_MASK, _box_union, _is_leaf, _pair_refs, _random_part, _shadow_root,
                                   _walk, compose_restate, compose_shadow, root_axis)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STACK = 64


class Part:
    """one part of a composed scene: nodes (offsets local to the part), primitive records, triangle and material counts,
    and its shadow tree: `shadow` its [n_prims - 1, 16] pairs, `single` the vertex box of its only primitive, `depth`
    its levels (0: it has none)"""

    def __init__(self, nodes, prims, n_tris, n_materials, shadow=None, single=None, depth=0):
        self.nodes, self.prims, self.n_tris, self.n_materials = nodes, prims, n_tris, n_materials
        self.shadow, self.single, self.depth = shadow, single, depth


def mesh_part(nodes, order, materials, n_materials, shadow=None, single=None, depth=0):
    """a mesh as trace_scene_upload_mesh_device builds it: prims[k] = {TRIANGLE, order[k], material[order[k]], order[k]}"""
    from trace_jl_b200 import _lib as tl
    order = np.asarray(order, np.uint32)
    prims = np.zeros(len(order), tl.prim_dtype)
    prims["kind"] = tl.PRIM_TRIANGLE
    prims["index"] = order
    prims["material"] = np.asarray(materials, np.uint32)[order]
    prims["original"] = order
    return Part(nodes, prims, len(order), n_materials, shadow, single, depth)


def compose_parts(a, b):
    """C(a, b): a new root, a's tree as first child, b's as second, b's records after a's with every reference shifted"""
    from trace_jl_b200 import _lib as tl
    na, pa = len(a.nodes), len(a.prims)
    nodes = np.zeros(1 + na + len(b.nodes), tl.node_dtype)
    part = a.nodes.copy()
    part["offset"] += np.where(_is_leaf(part), 0, 1).astype(np.uint32)
    nodes[1:1 + na] = part
    part = b.nodes.copy()
    part["offset"] += np.where(_is_leaf(part), pa, 1 + na).astype(np.uint32)
    nodes[1 + na:] = part
    lo, hi = _box_union(a.nodes[0]["bmin"], a.nodes[0]["bmax"], b.nodes[0]["bmin"], b.nodes[0]["bmax"])
    axis = root_axis(a.nodes[0], b.nodes[0])
    nodes[0] = (lo, hi, 1 + na, axis << 30)
    bp = b.prims.copy()
    bp["index"] += np.uint32(a.n_tris)
    bp["material"] += np.uint32(a.n_materials)
    bp["original"] += np.uint32(pa)
    shadow, depth = None, 0
    if a.depth and b.depth:
        shadow, depth = compose_shadow(a.shadow, b.shadow, axis, a.single, b.single), 1 + max(a.depth, b.depth)
    return Part(nodes, np.concatenate([a.prims, bp]), a.n_tris + b.n_tris, a.n_materials + b.n_materials, shadow, None,
                depth)


def group(meshes, lo=0, hi=None):
    """G(lo, hi): mesh lo when hi - lo == 1, else C(G(lo, mid), G(mid, hi)) with mid = lo + ceil((hi - lo) / 2)"""
    hi = len(meshes) if hi is None else hi
    if hi - lo == 1:
        return meshes[lo]
    mid = lo + (hi - lo + 1) // 2
    return compose_parts(group(meshes, lo, mid), group(meshes, mid, hi))


def compose_meshes(base, meshes):
    """D = C(base, G(0, k)) as a Part; its shadow tree is None unless every part has one and it is at most 64 levels"""
    d = compose_parts(base, group(meshes))
    if d.depth > STACK:
        d.shadow, d.depth = None, 0
    return d


def top_levels(k):
    """ceil(log2 k): the levels of G above its deepest mesh"""
    return int(np.ceil(np.log2(k))) if k > 1 else 0


# ------------------------------------------------------------------ hand-made parts
def _hand_shadow(rng, n):
    """a valid shadow tree over n primitives (random boxes, a balanced split of the slots, pairs in preorder from the
    root at 0): -> (pairs or None, single box, depth)"""
    if n == 1:
        return None, ([0.0, 0.0, 0.0], [1.0, 1.0, 1.0]), 1
    pairs = rng.random((n - 1, 16)).astype(np.float32)
    u = pairs.view(np.uint32)
    nxt = [0]

    def build(lo, hi):                                    # -> (reference, levels)
        if hi - lo == 1:
            return REF_LEAF | lo, 1
        me = nxt[0]
        nxt[0] += 1
        mid = (lo + hi) // 2
        (ra, da), (rb, db) = build(lo, mid), build(mid, hi)
        u[me, 6], u[me, 14], u[me, 7], u[me, 15] = ra, rb, 1, 0
        return me, 1 + max(da, db)

    return pairs, None, build(0, n)[1]


def _base_part(T, rng, nb, m, shadow=True):
    bn, border = _random_part(rng, nb, m, 10.0, 0.0)
    bprims = np.zeros(nb, T._lib.prim_dtype)
    bprims["index"], bprims["material"], bprims["original"] = border, 0, border
    sh, single, depth = _hand_shadow(rng, nb) if shadow else (None, None, 0)
    return Part(bn, bprims, nb, 2, sh, single, depth)


def _mesh_parts(rng, sizes, m):
    out = []
    for j, n in enumerate(sizes):
        mn, morder = _random_part(rng, n, m, 3.0, np.array([0.0, 20.0 + 5 * j, 0.0]))
        sh, single, depth = _hand_shadow(rng, n)
        out.append(mesh_part(mn, morder, rng.integers(0, 3, n), 3, sh, single, depth))
    return out


@pytest.mark.parametrize("nb, n, m", [(1, 1, 1), (1, 7, 1), (9, 1, 4), (40, 33, 1), (200, 150, 4)])
def test_one_mesh_is_the_single_attach(T, nb, n, m):
    rng = np.random.default_rng(nb * 1000 + n)
    base = _base_part(T, rng, nb, m)
    mesh = _mesh_parts(rng, [n], m)[0]
    d = compose_meshes(base, [mesh])
    order = mesh.prims["original"]
    nodes, prims = compose_restate(base.nodes, base.prims, base.n_tris, base.n_materials, mesh.nodes, order,
                                   np.asarray(mesh.prims["material"])[np.argsort(order)])
    assert nodes.tobytes() == d.nodes.tobytes() and prims.tobytes() == d.prims.tobytes()
    axis = int(nodes[0]["meta"]) >> 30
    assert d.shadow.tobytes() == compose_shadow(base.shadow, mesh.shadow, axis, base.single, mesh.single).tobytes()


@pytest.mark.parametrize("sizes, m", [([1, 1], 1), ([2, 1, 5], 1), ([3, 8, 1, 2, 40], 4), ([5] * 8, 1),
                                      ([1, 9, 2, 30, 4, 1, 7, 3, 11], 2)])
def test_restatement_invariants(T, sizes, m):
    rng = np.random.default_rng(len(sizes) * 100 + sum(sizes))
    nb = 17
    base = _base_part(T, rng, nb, m)
    meshes = _mesh_parts(rng, sizes, m)
    d = compose_meshes(base, meshes)
    k, total = len(sizes), nb + sum(sizes)
    seen, slots, _ = _walk(d.nodes)
    assert sorted(seen) == list(range(len(d.nodes)))          # preorder, every node reached once
    assert sorted(slots) == list(range(total))                # each primitive exactly once
    assert len(d.nodes) == 1 + nb_nodes(base) + (k - 1) + sum(len(p.nodes) for p in meshes)
    # mesh j's primitives: slots, triangles and `original` after the base's and meshes 0 .. j - 1's
    start, mat0 = nb, base.n_materials
    for p, n in zip(meshes, sizes):
        part = d.prims[start:start + n]
        assert np.array_equal(part["original"], start + p.prims["original"])
        assert np.array_equal(part["index"], start + p.prims["index"])
        assert np.array_equal(part["material"], mat0 + p.prims["material"])
        start, mat0 = start + n, mat0 + p.n_materials
    # every leaf of a mesh's part holds only that mesh's slots
    leaf = _is_leaf(d.nodes)
    off = d.nodes["offset"]
    assert (off[1:1 + nb_nodes(base)][leaf[1:1 + nb_nodes(base)]] < nb).all()
    # the shadow tree: n_prims - 1 pairs, every pair but the root referenced once, every slot once; its depth
    assert d.shadow is not None and len(d.shadow) == total - 1
    a, b = _pair_refs(d.shadow)
    refs = np.concatenate([a, b])
    assert sorted(refs[refs < REF_LEAF]) == list(range(1, total - 1))
    assert sorted(refs[refs >= REF_LEAF] & REF_MASK) == list(range(total))
    assert d.depth == _shadow_depth(d.shadow)
    assert d.depth <= 1 + max(base.depth, top_levels(k) + max(p.depth for p in meshes))
    # its root halves: the base's root box and reference, then G's (pair nb, after the base's nb - 1), with the node
    # tree's split axis
    u = d.shadow.view(np.uint32)
    assert u[0, 7] == 1 << (int(d.nodes[0]["meta"]) >> 30) and u[0, 15] == 0
    assert (u[0, 6], u[0, 14]) == (1, nb)
    lo, hi = _shadow_root(base.shadow, base.single)
    assert np.array_equal(d.shadow[0, 0:3], lo) and np.array_equal(d.shadow[0, 3:6], hi)


def nb_nodes(p):
    return len(p.nodes)


def _shadow_depth(pairs):
    u = pairs.view(np.uint32)
    best, stack = 0, [(0, 1)]
    while stack:
        i, dd = stack.pop()
        best = max(best, dd + 1)
        for col in (6, 14):
            r = int(u[i, col])
            if not r & REF_LEAF:
                stack.append((r, dd + 1))
    return best


def test_group_layout_is_balanced_in_slot_order(T):
    rng = np.random.default_rng(9)
    base = _base_part(T, rng, 5, 1)
    meshes = _mesh_parts(rng, [1] * 5, 1)
    d = compose_meshes(base, meshes)
    # G(0, 5) = C(G(0, 3), G(3, 5)), G(0, 3) = C(C(m0, m1), m2): group nodes right after the base, then in preorder
    nb = len(base.nodes)
    g = 1 + nb
    assert not _is_leaf(d.nodes[g:g + 1]).any() and int(d.nodes[g]["offset"]) == g + 1 + 2 + 3
    assert not _is_leaf(d.nodes[g + 1:g + 3]).any() and _is_leaf(d.nodes[g + 3:g + 5]).all()
    leaves = [int(d.nodes[i]["offset"]) for i in range(g, len(d.nodes)) if _is_leaf(d.nodes[i:i + 1])[0]]
    assert leaves == [5, 6, 7, 8, 9]                              # the meshes' slots in slot order


def test_shadow_depth_rule(T):
    rng = np.random.default_rng(2)
    base = _base_part(T, rng, 3, 1)
    meshes = _mesh_parts(rng, [2, 2, 2, 2], 1)
    meshes[1].depth = STACK - top_levels(4)                       # the deepest a new mesh may be with k = 4
    d = compose_meshes(base, meshes)
    assert d.shadow is None and d.depth == 0                     # 1 + 2 + 62 levels: no composed shadow tree
    meshes[1].depth = STACK - top_levels(4) - 1
    assert compose_meshes(base, meshes).depth == STACK
    meshes[2].depth = 0                                           # a part without a shadow tree: none composed
    assert compose_meshes(base, meshes).shadow is None


# ------------------------------------------------------------------ binding and argument checks
def test_binding_matches_header(T):
    txt = open(os.path.join(ROOT, "include", "trace_cuda.h")).read()
    m = re.search(r"int trace_scene_attach_meshes_device\((.*?)\);", txt, re.S)
    assert m and [" ".join(a.split()) for a in m.group(1).split(",")] == [
        "trace_ctx* ctx", "int64_t n_meshes", "const trace_mesh_device_desc* const* meshes", "int64_t* n_nodes_out"]
    res, args = T._lib.SIGNATURES["trace_scene_attach_meshes_device"]
    assert res is C.c_int and args[0] is C.c_void_p and args[1] is C.c_int64 and args[3] == C.POINTER(C.c_int64)
    assert args[2] == C.POINTER(C.POINTER(T._lib.MeshDeviceDesc))
    assert hasattr(T._lib.load(), "trace_scene_attach_meshes_device")


def _small_scene(T):
    m = T.MatteMaterial(T.ConstantTexture(T.RGBSpectrum(0.5)), T.ConstantTexture(0.0))
    core = T.ShapeCore(T.Transformation(), False)
    tris = T.create_triangle_mesh(core, 1, [1, 2, 3], 3, [(-1, -1, -3), (1, -1, -3), (0, 1, -3)])
    return T.Scene([], T.BVHAccel([T.GeometricPrimitive(t, m) for t in tris], 1))


def _mesh_stub(T, n, lo=(0, 0, 0), hi=(1, 2, 3)):
    """a DeviceMeshScene as far as CompositeScene and Context.upload look at it (making a real one needs a GPU)"""
    mesh = object.__new__(T.DeviceMeshScene)
    mesh.n_tris, mesh.lights = n, []
    mesh.bound = T.Bounds3(list(lo), list(hi))
    mesh.desc = lambda device: (T._lib.MeshDeviceDesc(), None)
    return mesh


def test_composite_scene_argument_checks(T):
    scene = _small_scene(T)
    with pytest.raises(ValueError, match="between 1 and 64 DeviceMeshScenes, got 0"):
        T.CompositeScene(scene, [])
    with pytest.raises(ValueError, match="between 1 and 64 DeviceMeshScenes, got 65"):
        T.CompositeScene(scene, [_mesh_stub(T, 1)] * 65)
    with pytest.raises(ValueError, match=r"mesh must be a DeviceMeshScene, got Scene \(mesh 1\)"):
        T.CompositeScene(scene, [_mesh_stub(T, 1), scene])
    with pytest.raises(ValueError, match=r"mesh must hold at least one triangle \(mesh 2\)"):
        T.CompositeScene(scene, (_mesh_stub(T, 1), _mesh_stub(T, 2), _mesh_stub(T, 0)))
    a, b = _mesh_stub(T, 3), _mesh_stub(T, 4, (-5, 0, 0), (0, 9, 1))
    cs = T.CompositeScene(scene, [a, b])
    assert cs.meshes == (a, b) and cs.mesh is None and not cs.has_unshaded
    assert cs.bound == scene.bound.union(a.bound).union(b.bound)
    one = T.CompositeScene(scene, a)
    assert one.meshes == (a,) and one.mesh is a
    assert T.CompositeScene(scene, mesh=a).meshes == (a,)                # the single-mesh keyword still works
    assert T.CompositeScene(scene, (m for m in [a, b])).meshes == (a, b)   # any iterable of meshes
    with pytest.raises(ValueError, match="mesh must be a DeviceMeshScene, got int"):
        T.CompositeScene(scene, 3)
    assert len(T.CompositeScene(scene, [a] * 64).meshes) == 64


class _StubLib:
    """the two library calls Context.upload makes for a CompositeScene, recorded: which descriptors are NULL"""

    def __init__(self):
        self.calls = []

    def trace_scene_upload(self, h, d):
        self.calls.append("upload")
        return 0

    def trace_scene_attach_meshes_device(self, h, n, arr, n_nodes):
        self.calls.append([bool(arr[j]) for j in range(n)])
        return 0


def test_upload_caches_each_slot(T, monkeypatch):
    import torch

    class _Stream:
        def synchronize(self):
            pass

    monkeypatch.setattr(torch.cuda, "current_stream", lambda device=None: _Stream())
    ctx = object.__new__(T.Context)
    ctx.lib, ctx.h, ctx.device = _StubLib(), C.c_void_p(), 0
    ctx._scene, ctx._n_nodes, ctx._base, ctx._meshes = None, 0, None, []
    env = _small_scene(T)
    m = [_mesh_stub(T, 1 + j) for j in range(4)]
    ctx.upload(T.CompositeScene(env, m[:3]))
    assert ctx.lib.calls == ["upload", [True, True, True]]
    ctx.upload(T.CompositeScene(env, m[:3]))                       # nothing changed: no call
    assert len(ctx.lib.calls) == 2
    new = _mesh_stub(T, 9)
    ctx.upload(T.CompositeScene(env, [m[0], new, m[2]]))          # one object replaced: one descriptor
    assert ctx.lib.calls[-1] == [False, True, False]
    ctx.upload(T.CompositeScene(env, [m[0], new, m[2], m[3]]))    # appended
    assert ctx.lib.calls[-1] == [False, False, False, True]
    ctx.upload(T.CompositeScene(env, [m[0]]))                     # shrunk: all kept
    assert ctx.lib.calls[-1] == [False] and ctx._mesh is m[0]
    ctx.upload(T.CompositeScene(env, [m[1], m[0]]))               # slot 0 holds another object now
    assert ctx.lib.calls[-1] == [True, True]
    env2 = _small_scene(T)
    ctx.upload(T.CompositeScene(env2, [m[1], m[0]]))              # a new environment clears every slot
    assert ctx.lib.calls[-2:] == ["upload", [True, True]]
    with pytest.raises(ValueError, match="not the one uploaded"):
        ctx.refit(T.CompositeScene(env2, [m[1]]), np.zeros((0, 3, 3), np.float32))
