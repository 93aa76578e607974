"""BVHAccel(..., builder="lbvh") from the host side: it needs a GPU and says so; the builder name is still checked; and
the numpy restatement of the tree (test_gpu_lbvh.lbvh_restate) has the shape the GPU build is held to."""
import numpy as np
import pytest

from test_bvh_build import _tree_depth
from test_gpu_lbvh import caustic_bounds, deep_bounds, lbvh_restate, one_centroid_bounds


def _prims(T, n=50):
    rng = np.random.default_rng(1)
    v = rng.uniform(-1, 1, (3 * n, 3)).astype(np.float32)
    core = T.ShapeCore(T.Transformation(), False)
    mesh = T.TriangleMesh(core.object_to_world, n, np.arange(1, 3 * n + 1, dtype=np.uint32), 3 * n, v)
    return [T.PrimitiveBatch(T.TriangleSet(core, mesh), None)]


def test_lbvh_builder_needs_a_gpu(T):
    """No CPU fallback: without a CUDA device the GPU build raises and says why (on a GPU box it builds the tree)."""
    import torch
    if torch.cuda.is_available():
        bvh = T.BVHAccel(_prims(T), 1, builder="lbvh")
        assert len(bvh.nodes) == 2 * 50 - 1 and sorted(bvh.order.tolist()) == list(range(50))
    else:
        with pytest.raises(RuntimeError, match="no CUDA device.*there is no CPU fallback"):
            T.BVHAccel(_prims(T), 1, builder="lbvh")


def test_unknown_builder_raises(T):
    with pytest.raises(ValueError):
        T.BVHAccel(_prims(T), 1, builder="octree")


def test_lbvh_restatement_shape(T):
    """Depths the specification implies: 1 000 equal centroids split by position (11 levels); the deep input is 67
    levels (65 with 4-primitive leaves), over the traversal stack's 64; the caustic mesh gives 2n - 1 nodes, depth 27."""
    nodes, order, depth = lbvh_restate(one_centroid_bounds(), 1)
    assert depth == _tree_depth(nodes) == 11 and len(nodes) == 1999
    assert lbvh_restate(deep_bounds(), 1)[2] == 67 and lbvh_restate(deep_bounds(), 4)[2] == 65
    nodes, order, depth = lbvh_restate(caustic_bounds(T), 1)
    assert len(nodes) == 176131 and depth == _tree_depth(nodes) == 27
    assert sorted(order.tolist()) == list(range(88066))
