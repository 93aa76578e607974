"""The opt-in GPU tree (trace_bvh_build_gpu, csrc/bvh_gpu.cu; BVHAccel(..., builder="lbvh")).  `lbvh_restate` states
the tree in numpy - Morton keys of the centroids, a stable sort, the binary radix tree's splits, preorder layout,
Julia min / max boxes - and the GPU build must reproduce it bit for bit.  On the GPU the tree must also give the
reference tree's closest hits (ties of equal t aside) with fewer box tests, and the same images."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib
from test_bvh_build import _tree_depth, random_bounds
from test_gpu_parity import camera_rays, image_report

pytestmark = pytest.mark.gpu

_SPREAD = ((32, 0x1F00000000FFFF), (16, 0x1F0000FF0000FF), (8, 0x100F00F00F00F00F), (4, 0x10C30C30C30C30C3),
           (2, 0x1249249249249249))


def _spread(q):
    x = q.astype(np.uint64) & np.uint64(0x1FFFFF)
    for shift, mask in _SPREAD:
        x = (x | (x << np.uint64(shift))) & np.uint64(mask)
    return x


def _high_bit(x):
    """index of the highest set bit of each (nonzero) uint64"""
    x = x.astype(np.uint64)
    h = np.zeros(len(x), np.int64)
    for s in (32, 16, 8, 4, 2, 1):
        t = x >> np.uint64(s)
        nz = t != 0
        h += np.where(nz, s, 0)
        x = np.where(nz, t, x)
    return h


def _jl_key(f):
    """float32 -> uint32 in Julia's order of min / max (-0.0 < +0.0; no NaN here)"""
    u = np.ascontiguousarray(f, np.float32).view(np.uint32)
    return np.where(u & np.uint32(0x80000000), ~u, u | np.uint32(0x80000000)).astype(np.uint32)


def _jl_float(k):
    u = np.where(k & np.uint32(0x80000000), k & np.uint32(0x7FFFFFFF), ~k).astype(np.uint32)
    return u.view(np.float32)


def lbvh_restate(bounds, max_node_primitives=1):
    """-> (nodes, order, depth): the tree trace_bvh_build_gpu specifies (include/trace_cuda.h), level by level."""
    from trace_jl_b200 import _lib as tl
    b = np.ascontiguousarray(bounds, np.float32)
    n, m = len(b), min(max(int(max_node_primitives), 1), 255)
    c = (np.float32(0.5) * b[:, :3] + np.float32(0.5) * b[:, 3:]).astype(np.float32)
    lo, hi = c.min(0), c.max(0)               # (the sign of a zero bound cannot change a key)
    ext = (hi - lo).astype(np.float32)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        s = np.where(ext > 0, np.float32(2097152.0) / ext, np.float32(0)).astype(np.float32)
        v = ((c - lo).astype(np.float32) * s).astype(np.float32)
        q = np.where(v >= 2097151, 2097151, np.where(v > 0, np.floor(v), 0)).astype(np.uint32)
    key = (_spread(q[:, 0]) << np.uint64(2)) | (_spread(q[:, 1]) << np.uint64(1)) | _spread(q[:, 2])
    order = np.argsort(key, kind="stable").astype(np.uint32)
    K = key[order]
    # top-down, one level at a time: ranges [A, B] of sorted positions
    levels = []
    A, B = np.zeros(1, np.int64), np.full(1, n - 1, np.int64)
    while len(A):
        cnt = B - A + 1
        inner = cnt > m
        a, bb = A[inner], B[inner]
        x = K[a] ^ K[bb]
        diff = x != 0
        hk = _high_bit(np.where(diff, x, 1))
        hp = _high_bit(np.where(diff, 1, (a ^ bb).astype(np.uint64)))
        prefix = (K[bb] >> hk.astype(np.uint64)) << hk.astype(np.uint64)
        sp = np.where(diff, np.searchsorted(K, prefix, "left") - 1, ((bb >> hp) << hp) - 1)
        axis = np.zeros(len(A), np.uint32)
        axis[inner] = np.where(diff, 2 - hk % 3, 0)
        levels.append(dict(A=A, B=B, inner=inner, axis=axis))
        A = np.stack([a, sp + 1], 1).reshape(-1)          # children: left, right of each interior node, in order
        B = np.stack([sp, bb], 1).reshape(-1)
    # bottom-up: emitted subtree sizes and boxes (as Julia-order keys)
    for li in range(len(levels) - 1, -1, -1):
        L = levels[li]
        size = np.ones(len(L["A"]), np.int64)
        box = np.empty((len(L["A"]), 6), np.uint32)
        leaf = ~L["inner"]
        la, lb = L["A"][leaf], L["B"][leaf]
        lk = np.stack([np.full(len(la), 0xFFFFFFFF, np.uint32)] * 3 + [np.zeros(len(la), np.uint32)] * 3, 1)
        for j in range(m):
            ok = la + j <= lb
            pk = _jl_key(b[order[np.minimum(la + j, n - 1)]])
            lk[:, :3] = np.where(ok[:, None], np.minimum(lk[:, :3], pk[:, :3]), lk[:, :3])
            lk[:, 3:] = np.where(ok[:, None], np.maximum(lk[:, 3:], pk[:, 3:]), lk[:, 3:])
        box[leaf] = lk
        if L["inner"].any():
            C_ = levels[li + 1]
            cs, cb = C_["size"].reshape(-1, 2), C_["box"].reshape(-1, 2, 6)
            size[L["inner"]] = 1 + cs[:, 0] + cs[:, 1]
            box[L["inner"]] = np.concatenate([np.minimum(cb[:, 0, :3], cb[:, 1, :3]), np.maximum(cb[:, 0, 3:], cb[:, 1, 3:])], 1)
        L["size"], L["box"] = size, box
    # top-down: preorder slots (left child = parent + 1, right child = parent + 1 + size(left))
    nodes = np.zeros(int(levels[0]["size"][0]), tl.node_dtype)
    pre = np.zeros(1, np.int64)
    for li, L in enumerate(levels):
        leaf = ~L["inner"]
        rec = nodes[pre]
        rec["bmin"], rec["bmax"] = _jl_float(L["box"][:, :3]), _jl_float(L["box"][:, 3:])
        if li + 1 < len(levels):
            cs = levels[li + 1]["size"].reshape(-1, 2)
            p = pre[L["inner"]]
            child_pre = np.stack([p + 1, p + 1 + cs[:, 0]], 1).reshape(-1)
        off = np.where(leaf, L["A"], 0)
        if L["inner"].any():
            off[L["inner"]] = child_pre.reshape(-1, 2)[:, 1]
        rec["offset"] = off
        rec["meta"] = np.where(leaf, tl.NODE_LEAF | (L["B"] - L["A"] + 1), L["axis"].astype(np.int64) << 30)
        nodes[pre] = rec
        if li + 1 < len(levels):
            pre = child_pre
    return nodes, order, len(levels)


def gpu_build(bounds, max_prims=1, device=0):
    """-> (rc, nodes, order); nodes / order are None when rc != 0 (and then no handle may come back)"""
    from trace_jl_b200 import _lib as tl
    lib = tl.load()
    bounds = np.ascontiguousarray(bounds, np.float32)
    h = C.c_void_p()
    rc = lib.trace_bvh_build_gpu(device, tl.ptr(bounds), len(bounds), max_prims, C.byref(h))
    if rc != 0:
        assert not h.value
        return rc, None, None
    nodes = np.zeros(lib.trace_bvh_num_nodes(h), tl.node_dtype)
    order = np.zeros(lib.trace_bvh_num_prims(h), np.uint32)
    lib.trace_bvh_copy(h, tl.ptr(nodes), tl.ptr(order))
    lib.trace_bvh_free(h)
    return rc, nodes, order


def clustered_bounds(n=200_000, seed=3):
    rng = np.random.default_rng(seed)
    c = rng.normal(size=(n, 3)).astype(np.float32) * np.array([40, 3, 15], np.float32) + rng.integers(0, 4, (n, 1)).astype(np.float32) * 30
    e = rng.uniform(0.0, 0.4, (n, 3)).astype(np.float32)
    e[rng.uniform(size=n) < 0.1] = 0
    return np.ascontiguousarray(np.concatenate([c - e, c + e], 1), dtype=np.float32)


def signed_zero_bounds(n=70_000, seed=11):
    """boxes with faces at +0.0 / -0.0 (the input of test_builder_signed_zeros_and_nan_bounds)"""
    rng = np.random.default_rng(seed)
    b = random_bounds(rng, n)
    z = rng.uniform(size=(n, 6)) < 0.15
    b[z] = np.where(rng.uniform(size=int(z.sum())) < 0.5, np.float32(0.0), np.float32(-0.0))
    return np.concatenate([np.minimum(b[:, :3], b[:, 3:]), np.maximum(b[:, :3], b[:, 3:])], 1).astype(np.float32)


def one_centroid_bounds(n=1000, seed=5):
    """boxes of different extents around one centroid (exact in float32): every key is equal, the splits go by position"""
    e = (np.random.default_rng(seed).integers(0, 1000, (n, 3)) / 1024.0).astype(np.float32)
    c = np.array([1, 2, 3], np.float32)
    return np.concatenate([c - e, c + e], 1).astype(np.float32)


def deep_bounds():
    """69 point boxes whose radix tree is 67 levels deep (65 with 4-primitive leaves): a far corner, five points at the
    origin, and 2^k on each axis for k = 0..20"""
    pts = [np.full(3, 2.0 ** 21)] + [np.zeros(3)] * 5
    for ax in range(3):
        for k in range(21):
            p = np.zeros(3)
            p[ax] = 2.0 ** k
            pts.append(p)
    p = np.array(pts, np.float32)
    return np.concatenate([p, p], 1)


def caustic_bounds(T):
    if not os.path.exists(T.scenes.ASSET_PLY):
        pytest.skip("asset missing")
    return T.scenes._caustic_bvh(1.25).prim_bounds


def same_bits(a, b):
    return a.tobytes() == b.tobytes()


INPUTS = {
    "caustic": caustic_bounds,
    "clustered_200k": lambda T: clustered_bounds(),
    "signed_zeros": lambda T: signed_zero_bounds(),
    "one_centroid": lambda T: one_centroid_bounds(),
    "n1": lambda T: np.array([[0, 1, 2, 3, 4, 5]], np.float32),
    "n2": lambda T: np.array([[0, 0, 0, 1, 1, 1], [-1, -1, -1, 0, 0, 0]], np.float32),
}


@pytest.mark.parametrize("name", sorted(INPUTS))
@pytest.mark.parametrize("max_prims", [1, 4])
def test_lbvh_bit_identical_to_restatement(T, name, max_prims):
    bounds = INPUTS[name](T)
    rc, nodes, order = gpu_build(bounds, max_prims)
    assert rc == 0
    rnodes, rorder, depth = lbvh_restate(bounds, max_prims)
    assert len(nodes) == len(rnodes) and same_bits(order, rorder)
    diff = np.nonzero(nodes.view(np.uint32).reshape(len(nodes), 8) != rnodes.view(np.uint32).reshape(len(nodes), 8))[0]
    assert len(diff) == 0, f"first differing node {diff[0]}: {nodes[diff[0]]} vs {rnodes[diff[0]]}"
    assert _tree_depth(nodes) == depth
    if name == "one_centroid" and max_prims == 1:
        assert depth == 11


def test_lbvh_deterministic(T):
    bounds = clustered_bounds()
    _, n1, o1 = gpu_build(bounds, 1)
    _, n2, o2 = gpu_build(bounds, 1)
    assert same_bits(n1, n2) and same_bits(o1, o2)


def test_lbvh_structure_caustic(T):
    bounds = caustic_bounds(T)
    n = len(bounds)
    rc, nodes, order = gpu_build(bounds, 1)
    assert rc == 0 and n == 88066
    assert len(nodes) == 2 * n - 1 == 176131 and _tree_depth(nodes) == 27
    assert sorted(order.tolist()) == list(range(n))
    covered = np.zeros(n, np.int64)
    meta = nodes["meta"].astype(np.int64)
    leaf = (meta >> 30) == 3
    for off, cnt in zip(nodes["offset"][leaf].astype(np.int64), meta[leaf] & 0x3FFFFFFF):
        covered[off:off + cnt] += 1
    assert (covered == 1).all()
    inner = np.nonzero(~leaf)[0]
    for ch in (inner + 1, nodes["offset"][inner].astype(np.int64)):
        assert (nodes["bmin"][ch] >= nodes["bmin"][inner]).all() and (nodes["bmax"][ch] <= nodes["bmax"][inner]).all()


def test_lbvh_refusals(T):
    b = random_bounds(np.random.default_rng(2), 100)
    b[17, 4] = np.nan
    assert gpu_build(b, 1)[0] == 5
    for m in (1, 4):
        assert gpu_build(deep_bounds(), m)[0] == 6
    # through BVHAccel: degenerate triangles at the same points
    pts = deep_bounds()[:, :3]
    core = T.ShapeCore(T.Transformation(), False)
    idx = np.repeat(np.arange(1, len(pts) + 1, dtype=np.uint32), 3)
    mesh = T.TriangleMesh(core.object_to_world, len(pts), idx, len(pts), pts)
    with pytest.raises(RuntimeError, match="deeper than 64 levels"):
        T.BVHAccel([T.PrimitiveBatch(T.TriangleSet(core, mesh), None)], 1, builder="lbvh")


def test_lbvh_same_hits_as_reference_tree(T, ctx):
    """As test_optin_sah_tree_on_gpu: 2e6 rays on the caustic mesh, t bit-identical to the reference tree's, the same
    primitive except on ties of equal t, fewer box tests; the oracle walking the same LBVH tree agrees bit for bit."""
    if not os.path.exists(T.scenes.ASSET_PLY):
        pytest.skip("asset missing")
    rng = np.random.default_rng(11)
    n = 2_000_000
    flats = {}
    for builder in ("reference", "lbvh"):
        scene, _, _ = T.scenes.caustic_glass(builder=builder)
        flats[builder] = (scene, scene.flatten())
    lo, hi = flats["reference"][1].nodes[0]["bmin"], flats["reference"][1].nodes[0]["bmax"]
    target = (lo + rng.random((n, 3), dtype=np.float32) * (hi - lo)).astype(np.float32)
    origin = np.where(rng.random((n, 1)) < 0.5, np.array([[0, 150, 150]], np.float32),
                      (target + rng.normal(size=(n, 3)).astype(np.float32) * 20)).astype(np.float32)
    d = (target - origin).astype(np.float32)
    out = {}
    for builder, (scene, flat) in flats.items():
        ctx.upload(scene)
        ctx.set_option("count_nodes", 1)
        ctx.reset_stats()
        out[builder] = ctx.intersect(origin, d) + (ctx.stats()["nodes_visited"],)
        ctx.set_option("count_nodes", 0)
    (pa, ta, ba, na), (pb, tb, bb, nb) = out["reference"], out["lbvh"]
    print("nodes visited per ray: reference", na / n, "lbvh", nb / n)
    assert (pa != 0).sum() > n // 4
    assert np.array_equal(ta.view(np.uint32), tb.view(np.uint32))
    assert (pa != pb).mean() < 1e-3
    assert nb < na
    m = 100_000
    op, ot, ob = oracle_lib.OracleScene(flats["lbvh"][1]).intersect(origin[:m], d[:m], slab=0)
    assert np.array_equal(op, pb[:m]) and np.array_equal(ot.view(np.uint32), tb[:m].view(np.uint32))
    assert np.array_equal(ob.view(np.uint32), bb[:m].view(np.uint32))


def test_lbvh_spheres_same_t(T, ctx):
    """Spheres (shadows scene): camera rays, which start outside every sphere, hit at bit-identical t on either tree."""
    scene, camera, _ = T.scenes.shadows(resolution=64)
    prims = [p for _, p in scene.aggregate.items]
    lscene = T.Scene(scene.lights, T.BVHAccel(prims, 1, builder="lbvh"))
    o, d = camera_rays(T, camera, 200_000, np.random.default_rng(4))
    ctx.upload(scene)
    pa, ta, _ = ctx.intersect(o, d)
    ctx.upload(lscene)
    pb, tb, _ = ctx.intersect(o, d)
    assert (pa != 0).mean() > 0.1
    assert np.array_equal(ta.view(np.uint32), tb.view(np.uint32))


def _whitted(T, ctx, builder):
    scene, camera, _ = T.scenes.tessellated(cells=48, stacks=26, slices=24, res=(160, 90), builder=builder)
    ctx.upload(scene)
    cam, fd = camera.pod(), camera.film.desc()
    film = np.zeros_like(camera.film.pixels)
    ctx.check(ctx.lib.trace_render_whitted(ctx.h, C.byref(cam), C.byref(fd), 4, 5, C.c_uint64(9), T._lib.ptr(film)))
    return film


def _sppm(T, ctx, builder):
    scene, camera, kw = T.scenes.caustic_glass(resolution=64, builder=builder)
    ctx.upload(scene)
    cam, fd = camera.pod(), camera.film.desc()
    h, w = camera.film.pixels.shape[:2]
    rgb = np.zeros((h, w, 3), np.float32)
    ctx.check(ctx.lib.trace_render_sppm(ctx.h, C.byref(cam), C.byref(fd), kw["initial_search_radius"], kw["max_depth"], 2,
                                        -1, 0, C.c_uint64(3), C.cast(None, T._lib.SPPM_CB), None, T._lib.ptr(rgb)))
    return np.concatenate([rgb, np.ones_like(rgb[..., :1])], -1)


def test_lbvh_images_match_reference_tree(T, ctx):
    a, b = _whitted(T, ctx, "reference"), _whitted(T, ctx, "lbvh")
    rel_mse, frac, werr = image_report(b, a, "whitted/tess-small lbvh-vs-reference tree")
    assert werr < 1e-5 and rel_mse < 1e-5 and frac > 0.998
    if not os.path.exists(T.scenes.ASSET_PLY):
        pytest.skip("asset missing")
    a, b = _sppm(T, ctx, "reference"), _sppm(T, ctx, "lbvh")
    rel_mse, frac, werr = image_report(b, a, "sppm/caustic_glass 64^2 lbvh-vs-reference tree")
    assert float(a[..., :3].max()) > 0
    assert werr < 1e-5 and rel_mse < 1e-5 and frac > 0.998
