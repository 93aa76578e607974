"""Hand-made scene descriptors through trace_scene_upload (-m gpu), checked exactly against the oracle walking the same
descriptor.  The upload derives the pair records, the last-of-leaf bits and the root reference from the node array;
these trees hold the node shapes the builders rarely or never emit: a zero-primitive leaf, "sphere below" references
on both children of a node, leaves whose last primitive is a sphere, and a one-node tree whose leaf does not start at
primitive 0."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib
from trace_jl_b200 import _lib
from trace_jl_b200.scene import FlatScene

pytestmark = pytest.mark.gpu

# the walks of tests/test_gpu_parity.py: (slab, walk, leaf_wait); slab 1 is not hit-equivalent and is not asserted there
WALKS = [(0, 0, 0), (2, 0, 0)] + [(s, 0, lw) for s, lw in ((2, 8), (2, 4), (0, 16), (2, 32), (2, 16), (0, 8))] + \
        [(0, 1, 0), (2, 1, 0)]


class HandScene(FlatScene):
    """The shapes, materials and lights of a flattened scene under a hand-made node array and primitive list.
    prims: ("t" | "s", index) in BVH slot order; nodes: preorder ("leaf", offset, count, box or None) or
    ("interior", axis, second child); None boxes are the union of the leaf's primitives, interior boxes the union of
    the children's."""

    def __init__(self, base, prims, nodes):
        self.__dict__.update(base.__dict__)
        if all(k == "t" for k, _ in prims):
            self.spheres = self.spheres[:0]      # no analytic sphere in the scene: the upload builds a shadow tree
        kind = {"t": _lib.PRIM_TRIANGLE, "s": _lib.PRIM_SPHERE}
        self.prims = np.zeros(len(prims), _lib.prim_dtype)
        for i, (k, idx) in enumerate(prims):
            self.prims[i] = (kind[k], idx, 0, i)
        pbox = [self._box(k, idx) for k, idx in prims]
        self.nodes = np.zeros(len(nodes), _lib.node_dtype)

        def fill(i):
            nd = nodes[i]
            if nd[0] == "leaf":
                _, off, cnt, box = nd
                if box is None:
                    box = (np.min([pbox[j][0] for j in range(off, off + cnt)], 0),
                           np.max([pbox[j][1] for j in range(off, off + cnt)], 0))
                self.nodes[i] = (box[0], box[1], off, 0xC0000000 | cnt)
                return box
            _, axis, second = nd
            a, b = fill(i + 1), fill(second)
            box = (np.minimum(a[0], b[0]), np.maximum(a[1], b[1]))
            self.nodes[i] = (box[0], box[1], second, axis << 30)
            return box

        fill(0)

    def _box(self, kind, idx):
        if kind == "t":
            v = self.tri_vertices[idx]
            return v.min(0), v.max(0)
        b = self.sphere_bounds[idx]
        return b[:3], b[3:]


@pytest.fixture(scope="module")
def base(T):
    return T.scenes.shadows(resolution=16)[0].flatten()


@pytest.fixture(scope="module")
def hctx(T):
    c = T.Context(0)                 # its own context: these uploads bypass Context.upload's scene cache
    yield c
    c.close()


def rays(scene, n, seed):
    rng = np.random.default_rng(seed)
    lo = scene.nodes[0]["bmin"].astype(np.float64)
    hi = scene.nodes[0]["bmax"].astype(np.float64)
    ext = np.maximum(hi - lo, 0.1)
    o = rng.uniform(lo - 2 * ext, hi + 2 * ext, (n, 3))
    tgt = rng.uniform(lo - 0.1 * ext, hi + 0.1 * ext, (n, 3))
    d = (tgt - o).astype(np.float32)
    tmax = np.where(rng.uniform(size=n) < 0.5, np.inf, rng.uniform(0.2, 1.2, n)).astype(np.float32)
    return o.astype(np.float32), d, tmax


def check(hctx, scene, label):
    d = scene.desc()
    hctx.check(hctx.lib.trace_scene_upload(hctx.h, C.byref(d)))
    osc = oracle_lib.OracleScene(scene)
    o, dr, tmax = rays(scene, 20000, 5)
    for tm in (None, tmax):
        rprim, rt, rb = osc.intersect(o, dr, tm, slab=0)
        rocc = osc.occluded(o, dr, tm, slab=0)
        assert np.count_nonzero(rprim) > 100 and np.count_nonzero(rocc) > 100, f"{label}: too few hits to say anything"
        for slab, walk, lw in WALKS:
            hctx.set_option("slab", slab)
            hctx.set_option("walk", walk)
            if lw:
                hctx.set_option("leaf_wait", lw)
            prim, t, b = hctx.intersect(o, dr, tm)
            occ = hctx.occluded(o, dr, tm)
            what = f"{label}/slab{slab}/walk{walk}/leaf_wait{lw}/tmax{'inf' if tm is None else 'finite'}"
            assert np.array_equal(prim, rprim), f"{what}: {np.count_nonzero(prim != rprim)} primitive ids differ"
            assert np.array_equal(t.view(np.uint32), rt.view(np.uint32)), f"{what}: t differs"
            assert np.array_equal(b.view(np.uint32), rb.view(np.uint32)), f"{what}: barycentrics differ"
            assert np.array_equal(occ, rocc), f"{what}: {np.count_nonzero(occ != rocc)} any-hit results differ"
    hctx.set_option("slab", 2)
    hctx.set_option("walk", 1)


def test_zero_primitive_leaf(hctx, base):
    # node 3 holds no primitive; its box is the empty one the builders give such a leaf (+inf, -inf), which fails every
    # slab test of the reference (a count of 0 would make it an interior node there, so it must never be entered)
    empty = (np.full(3, np.inf, np.float32), np.full(3, -np.inf, np.float32))
    scene = HandScene(base, [("t", 0), ("t", 1), ("t", 2), ("t", 3)],
                      [("interior", 0, 2), ("leaf", 0, 2, None), ("interior", 2, 4), ("leaf", 2, 0, empty),
                       ("leaf", 2, 2, None)])
    check(hctx, scene, "zero-primitive leaf")
    assert hctx.shadow_tree() is not None          # a triangle-only scene: any-hit rays of the pair walk take it


def test_sphere_below_both_children_and_sphere_last_in_leaf(hctx, base):
    # both children of the root and of node 1 have a sphere below; leaves 2 and 6 end with a sphere, leaf 5 has none
    scene = HandScene(base, [("t", 0), ("s", 0), ("s", 1), ("t", 1), ("t", 2), ("s", 2)],
                      [("interior", 1, 4), ("interior", 0, 3), ("leaf", 0, 2, None), ("leaf", 2, 2, None),
                       ("interior", 2, 6), ("leaf", 4, 1, None), ("leaf", 5, 1, None)])
    check(hctx, scene, "sphere below")


def test_single_leaf_not_at_slot_zero(hctx, base):
    # the root is a leaf over slots 2..4 (ending with a sphere); slots 0 and 1 belong to no leaf
    scene = HandScene(base, [("s", 3), ("s", 0), ("t", 0), ("t", 1), ("s", 1)], [("leaf", 2, 3, None)])
    check(hctx, scene, "single leaf at slot 2")
