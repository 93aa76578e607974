"""The mesh attach's host side, without a GPU (trace_scene_attach_mesh_device, csrc/upload_device.cu; CompositeScene +
Context.upload).  `compose_restate` and `compose_shadow` restate the composed scene D and its shadow tree in numpy:
tests/test_gpu_attach_mesh.py holds the device to them bit for bit, so their invariants are checked here on trees made
by hand.  Also: the ctypes binding against the header, and CompositeScene's argument checks."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from test_gpu_lbvh import _jl_float, _jl_key, lbvh_restate

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LEAF, REF_LEAF, REF_MASK = 0xC0000000, 0x80000000, 0x3FFFFFFF


def _is_leaf(nodes):
    return (nodes["meta"].astype(np.int64) >> 30) == 3


def _box_union(a_lo, a_hi, b_lo, b_hi):
    """Julia min / max (-0.0 < +0.0) of two boxes"""
    ka, kb = _jl_key(np.stack([a_lo, a_hi]).astype(np.float32)), _jl_key(np.stack([b_lo, b_hi]).astype(np.float32))
    return _jl_float(np.minimum(ka[0], kb[0])), _jl_float(np.maximum(ka[1], kb[1]))


def root_axis(base_root, mesh_root):
    """the k maximising (mesh.min[k] + mesh.max[k]) - (base.min[k] + base.max[k]) in float32; ties to the lowest k,
    non-finite values lose (0 when none is finite)"""
    with np.errstate(over="ignore", invalid="ignore"):
        v = ((mesh_root["bmin"] + mesh_root["bmax"]).astype(np.float32) -
             (base_root["bmin"] + base_root["bmax"]).astype(np.float32)).astype(np.float32)
    best = None
    for k in range(3):
        if np.isfinite(v[k]) and (best is None or v[k] > v[best]):
            best = k
    return 0 if best is None else best


def compose_restate(base_nodes, base_prims, n_base_tris, n_base_materials, mesh_nodes, mesh_order, mesh_materials):
    """-> (nodes, prims) of D: a new root over the base's tree (first child) and the mesh's LBVH (second child, as
    trace_scene_upload_mesh_device builds it: `mesh_nodes` with offsets local to the mesh, `mesh_order` its slot ->
    triangle map, `mesh_materials` the material of each mesh triangle)"""
    from trace_jl_b200 import _lib as tl
    nb, pb = len(base_nodes), len(base_prims)
    nodes = np.zeros(1 + nb + len(mesh_nodes), tl.node_dtype)
    part = base_nodes.copy()
    part["offset"] += np.where(_is_leaf(part), 0, 1).astype(np.uint32)
    nodes[1:1 + nb] = part
    part = mesh_nodes.copy()
    part["offset"] += np.where(_is_leaf(part), pb, 1 + nb).astype(np.uint32)
    nodes[1 + nb:] = part
    lo, hi = _box_union(base_nodes[0]["bmin"], base_nodes[0]["bmax"], mesh_nodes[0]["bmin"], mesh_nodes[0]["bmax"])
    nodes[0] = (lo, hi, 1 + nb, root_axis(base_nodes[0], mesh_nodes[0]) << 30)
    order = np.asarray(mesh_order, np.uint32)
    mesh = np.zeros(len(order), tl.prim_dtype)
    mesh["kind"] = tl.PRIM_TRIANGLE
    mesh["index"] = n_base_tris + order
    mesh["material"] = n_base_materials + np.asarray(mesh_materials, np.uint32)[order]
    mesh["original"] = pb + order
    return nodes, np.concatenate([base_prims, mesh])


def _pair_refs(pairs):
    u = pairs.view(np.uint32)
    return u[:, 6], u[:, 14]


def _shadow_root(pairs, box_of_single):
    """a shadow tree part's root box: the union of its pair 0's halves, or its single primitive's box"""
    if pairs is None or len(pairs) == 0:
        return box_of_single
    return _box_union(pairs[0, 0:3], pairs[0, [3, 4, 5]], pairs[0, 8:11], pairs[0, [11, 12, 13]])


def compose_shadow(base_pairs, mesh_pairs, axis, base_single_box=None, mesh_single_box=None):
    """-> D's composed shadow tree [n_prims - 1, 16] float32 from the two parts' own ([Pb - 1, 16] and [n - 1, 16];
    None or empty for a part of one primitive, whose vertex box is then given as (lo, hi))"""
    pb = 1 if base_pairs is None else len(base_pairs) + 1
    n = 1 if mesh_pairs is None else len(mesh_pairs) + 1
    out = np.zeros((pb + n - 1, 16), np.float32)
    u = out.view(np.uint32)

    def put(dst, src, shift_pair, shift_leaf):
        out[dst:dst + len(src)] = src
        for col in (6, 14):
            r = u[dst:dst + len(src), col]
            u[dst:dst + len(src), col] = np.where(r & REF_LEAF, REF_LEAF | ((r & REF_MASK) + shift_leaf), r + shift_pair)

    if pb > 1:
        put(1, base_pairs, 1, 0)
    if n > 1:
        put(pb, mesh_pairs, pb, pb)
    halves = [(_shadow_root(base_pairs, base_single_box), 1 if pb > 1 else REF_LEAF | 0, 1 << axis),
              (_shadow_root(mesh_pairs, mesh_single_box), pb if n > 1 else REF_LEAF | pb, 0)]
    for k, ((lo, hi), ref, extra) in enumerate(halves):
        out[0, 8 * k:8 * k + 6] = [lo[0], lo[1], lo[2], hi[0], hi[1], hi[2]]
        u[0, 8 * k + 6], u[0, 8 * k + 7] = ref, extra
    return out


# ------------------------------------------------------------------ invariants of the restatement
def _walk(nodes):
    """preorder walk from the root: -> (visited node ids, primitive slots the leaves hold, max depth)"""
    seen, slots, depth = [], [], 0
    stack = [(0, 1)]
    while stack:
        i, d = stack.pop()
        seen.append(i)
        depth = max(depth, d)
        nd = nodes[i]
        if (int(nd["meta"]) >> 30) == 3:
            slots.extend(range(int(nd["offset"]), int(nd["offset"]) + (int(nd["meta"]) & 0x3FFFFFFF)))
        else:
            assert i + 1 < int(nd["offset"]) < len(nodes)
            stack += [(int(nd["offset"]), d + 1), (i + 1, d + 1)]
    return seen, slots, depth


def _random_part(rng, n, m, spread, shift):
    lo = (rng.random((n, 3)) * spread + shift).astype(np.float32)
    b = np.concatenate([lo, lo + rng.random((n, 3)).astype(np.float32)], 1).astype(np.float32)
    nodes, order, _ = lbvh_restate(b, m)
    return nodes, order


@pytest.mark.parametrize("nb, n, m", [(1, 1, 1), (1, 7, 1), (9, 1, 4), (40, 33, 1), (200, 150, 4)])
def test_restatement_invariants(T, nb, n, m):
    rng = np.random.default_rng(nb * 1000 + n)
    bn, border = _random_part(rng, nb, m, 10.0, 0.0)
    mn, morder = _random_part(rng, n, m, 3.0, np.array([0.0, 20.0, 0.0]))
    bprims = np.zeros(nb, T._lib.prim_dtype)
    bprims["index"], bprims["material"], bprims["original"] = border, 0, border
    mats = rng.integers(0, 3, n)
    nodes, prims = compose_restate(bn, bprims, nb, 2, mn, morder, mats)
    seen, slots, _ = _walk(nodes)
    assert sorted(seen) == list(range(len(nodes)))             # preorder, every node reached once
    assert sorted(slots) == list(range(nb + n))                # each primitive exactly once
    assert np.array_equal(prims["original"][nb:], nb + morder)
    assert np.array_equal(prims["index"][nb:], nb + morder) and np.array_equal(prims["material"][nb:], 2 + mats[morder])
    root, k = nodes[0], len(bn)
    assert int(root["offset"]) == 1 + k and (int(root["meta"]) >> 30) == 1          # the mesh lies above along y
    assert np.array_equal(root["bmin"], np.minimum(bn[0]["bmin"], mn[0]["bmin"]))
    assert np.array_equal(root["bmax"], np.maximum(bn[0]["bmax"], mn[0]["bmax"]))
    # leaves of the mesh part hold only mesh slots, the base's only base slots
    leaf = _is_leaf(nodes)
    assert (nodes["offset"][1:1 + k][leaf[1:1 + k]] < nb).all() and (nodes["offset"][1 + k:][leaf[1 + k:]] >= nb).all()


def test_root_axis_rule(T):
    box = lambda lo, hi: np.array((lo, hi, 0, LEAF | 1), T._lib.node_dtype)
    base = box([0, 0, 0], [1, 1, 1])
    assert root_axis(base, box([0, 0, 5], [1, 1, 6])) == 2
    assert root_axis(base, box([3, 3, 0], [4, 4, 1])) == 0           # a tie goes to the lowest axis
    assert root_axis(base, box([-5, -5, -5], [-4, -4, -4])) == 0     # all below: the largest difference, still a tie
    assert root_axis(base, box([-5, 1, -9], [-4, 2, -8])) == 1
    assert root_axis(base, box([0, 0, 0], [np.inf, 1, -1])) == 1     # inf loses
    assert root_axis(box([0, 0, 0], [np.inf, np.inf, np.inf]), box([0, 0, 0], [np.inf, np.inf, np.inf])) == 0


def test_shadow_composition_references(T):
    rng = np.random.default_rng(4)
    bp = rng.random((4, 16)).astype(np.float32)
    mp = rng.random((2, 16)).astype(np.float32)
    bu, mu = bp.view(np.uint32), mp.view(np.uint32)
    bu[:, 6], bu[:, 14] = [1, REF_LEAF | 0, 3, REF_LEAF | 2], [2, REF_LEAF | 1, REF_LEAF | 3, REF_LEAF | 4]
    mu[:, 6], mu[:, 14] = [1, REF_LEAF | 0], [REF_LEAF | 2, REF_LEAF | 1]
    out = compose_shadow(bp, mp, axis=2)
    a, b = _pair_refs(out)
    assert len(out) == 5 + 3 - 1
    assert (a[0], b[0]) == (1, 5) and out.view(np.uint32)[0, 7] == 4 and out.view(np.uint32)[0, 15] == 0
    assert list(a[1:5]) == [2, REF_LEAF | 0, 4, REF_LEAF | 2] and list(b[1:5]) == [3, REF_LEAF | 1, REF_LEAF | 3, REF_LEAF | 4]
    assert list(a[5:]) == [6, REF_LEAF | 5] and list(b[5:]) == [REF_LEAF | 7, REF_LEAF | 6]
    # every pair but the root is referenced once, every primitive slot once
    refs = np.concatenate([a, b])
    assert sorted(refs[refs < REF_LEAF]) == list(range(1, len(out)))
    assert sorted(refs[refs >= REF_LEAF] & REF_MASK) == list(range(len(out) + 1))
    single = compose_shadow(None, None, axis=0, base_single_box=([0, 0, 0], [1, 1, 1]), mesh_single_box=([2, 2, 2], [3, 3, 3]))
    assert len(single) == 1 and list(_pair_refs(single)[0]) == [REF_LEAF | 0] and list(_pair_refs(single)[1]) == [REF_LEAF | 1]


# ------------------------------------------------------------------ binding and argument checks
def test_binding_matches_header(T):
    txt = open(os.path.join(ROOT, "include", "trace_cuda.h")).read()
    m = re.search(r"int trace_scene_attach_mesh_device\((.*?)\);", txt, re.S)
    assert m and [a.strip() for a in m.group(1).split(",")] == [
        "trace_ctx* ctx", "const trace_mesh_device_desc* mesh", "int64_t* n_nodes_out"]
    res, args = T._lib.SIGNATURES["trace_scene_attach_mesh_device"]
    assert res is C.c_int and args[0] is C.c_void_p and args[2] == C.POINTER(C.c_int64)
    assert args[1] == C.POINTER(T._lib.MeshDeviceDesc)
    assert T._lib.SIGNATURES["trace_scene_upload_mesh_device"] == (res, args)
    assert hasattr(T._lib.load(), "trace_scene_attach_mesh_device")


def _small_scene(T):
    m = T.MatteMaterial(T.ConstantTexture(T.RGBSpectrum(0.5)), T.ConstantTexture(0.0))
    core = T.ShapeCore(T.Transformation(), False)
    tris = T.create_triangle_mesh(core, 1, [1, 2, 3], 3, [(-1, -1, -3), (1, -1, -3), (0, 1, -3)])
    return T.Scene([], T.BVHAccel([T.GeometricPrimitive(t, m) for t in tris], 1))


def _mesh_stub(T, n):
    """a DeviceMeshScene as far as CompositeScene looks at it (making a real one needs a GPU)"""
    mesh = object.__new__(T.DeviceMeshScene)
    mesh.n_tris, mesh.lights = n, []
    mesh.bound = T.Bounds3([0, 0, 0], [1, 2, 3])
    return mesh


def test_composite_scene_argument_checks(T):
    scene = _small_scene(T)
    with pytest.raises(ValueError, match="scene must be a Scene, got FlatScene"):
        T.CompositeScene(scene.flatten(), _mesh_stub(T, 3))
    with pytest.raises(ValueError, match="mesh must be a DeviceMeshScene, got Scene"):
        T.CompositeScene(scene, scene)
    with pytest.raises(ValueError, match="mesh must hold at least one triangle"):
        T.CompositeScene(scene, _mesh_stub(T, 0))
    cs = T.CompositeScene(scene, _mesh_stub(T, 3))
    assert cs.bound == scene.bound.union(T.Bounds3([0, 0, 0], [1, 2, 3])) and not cs.has_unshaded
