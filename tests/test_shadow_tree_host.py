"""The two facts the shadow-tree any-hit walk (traverse.cuh, traverse_shadow) rests on, checked without a GPU:
  * the lemma: when a triangle's vertex box is nested in a parent box and textbook-accepts a ray (t_enter <= t_exit,
    t_exit > 0, t_enter < t_max, on the six float32 slab products), the parent textbook-accepts with an entry <= the
    triangle box's - and so does the reference's literal test (bounds.jl:180-200, loose y far bound) with tx_min < t_max;
  * on the uploaded trees, every reference-tree box contains the vertex boxes of the primitives below it."""
import os

import numpy as np
import pytest

from test_refit_host import tess_small

f32 = np.float32


def products(lo, hi, o, inv):
    """float32 slab products, entry / exit per axis (no NaN: inv finite and non-zero)"""
    a = ((lo - o) * inv).astype(f32)
    b = ((hi - o) * inv).astype(f32)
    return np.minimum(a, b), np.maximum(a, b), a, b


def textbook(lo, hi, o, inv, tmax):
    e, x, _, _ = products(lo, hi, o, inv)
    t_enter, t_exit = e.max(1), x.min(1)
    return (t_enter <= t_exit) & (t_exit > 0) & (t_enter < tmax), t_enter


def literal(lo, hi, o, inv, tmax):
    """the reference's test as slab_test<0> writes it: sign-selected products, the y far bound keeps the LARGER value"""
    neg = inv < 0
    near = np.where(neg, hi, lo)
    far = np.where(neg, lo, hi)
    t0 = ((near - o) * inv).astype(f32)
    t1 = ((far - o) * inv).astype(f32)
    ax0, ay0, az0 = t0.T
    ax1, ay1, az1 = t1.T
    ok = ~((ax0 > ay1) | (ay0 > ax1))
    tmin = np.where(ay0 > ax0, ay0, ax0)
    tmx = np.where(ay1 > ax1, ay1, ax1)
    ok &= ~((tmin > az1) | (az0 > tmx))
    tmin = np.where(az0 > tmin, az0, tmin)
    tmx = np.where(az1 < tmx, az1, tmx)
    return ok & (tmin < tmax) & (tmx > 0), tmin


def check_lemma(lo, hi, plo, phi, o, d, tmax):
    with np.errstate(divide="ignore", over="ignore"):
        inv = (f32(1) / d).astype(f32)
    keep = np.isfinite(inv).all(1) & (inv != 0).all(1)
    lo, hi, plo, phi, o, inv, tmax = lo[keep], hi[keep], plo[keep], phi[keep], o[keep], inv[keep], tmax[keep]
    assert np.all(plo <= lo) and np.all(phi >= hi)
    with np.errstate(over="ignore", invalid="ignore"):
        return _check(lo, hi, plo, phi, o, inv, tmax)


def _check(lo, hi, plo, phi, o, inv, tmax):
    acc, te = textbook(lo, hi, o, inv, tmax)
    pacc, pte = textbook(plo, phi, o, inv, tmax)
    lacc, ltmin = literal(plo, phi, o, inv, tmax)
    assert np.all(pacc[acc]), "a parent of an accepted triangle box rejects"
    assert np.all(pte[acc] <= te[acc])
    assert np.all(lacc[acc]), "the reference's literal test rejects a parent of an accepted triangle box"
    assert np.all(ltmin[acc] == pte[acc])
    return int(acc.sum())


def random_case(rng, n):
    lo = rng.normal(size=(n, 3)).astype(f32)
    hi = (lo + np.abs(rng.normal(size=(n, 3))).astype(f32) * f32(0.1)).astype(f32)
    grow = lambda: (np.abs(rng.normal(size=(n, 3))) * (rng.random((n, 3)) < 0.6)).astype(f32)   # 40 %: a shared face
    plo = (lo - grow()).astype(f32)
    phi = (hi + grow()).astype(f32)
    o = (rng.normal(size=(n, 3)) * 3).astype(f32)
    tgt = (lo + (hi - lo) * rng.random((n, 3)).astype(f32)).astype(f32)
    d = (tgt - o).astype(f32)
    tmax = np.where(rng.random(n) < 0.5, np.inf, rng.uniform(0.5, 1.5, n)).astype(f32)
    return lo, hi, plo, phi, o, d, tmax


def test_lemma_random_boxes():
    rng = np.random.default_rng(1)
    accepted = check_lemma(*random_case(rng, 400_000))
    assert accepted > 100_000


def test_lemma_adversarial_boxes():
    """signed zeros in boxes and origins, zero-thickness boxes, boxes sharing faces with their parent, rays that start
    on a face or graze one, tiny and huge direction components"""
    rng = np.random.default_rng(2)
    n = 400_000
    grid = np.array([-1.0, -0.0, 0.0, 0.5, 1.0], f32)
    pick = lambda shape: grid[rng.integers(0, len(grid), shape)]
    a, b = pick((n, 3)), pick((n, 3))
    lo, hi = np.minimum(a, b), np.maximum(a, b)                   # many zero-thickness axes
    flat = rng.random((n, 3)) < 0.3
    hi = np.where(flat, lo, hi).astype(f32)
    plo = np.where(rng.random((n, 3)) < 0.5, lo, np.minimum(lo, pick((n, 3)))).astype(f32)
    phi = np.where(rng.random((n, 3)) < 0.5, hi, np.maximum(hi, pick((n, 3)))).astype(f32)
    o = np.where(rng.random((n, 3)) < 0.5, pick((n, 3)), rng.normal(size=(n, 3)) * 2).astype(f32)
    tgt = (lo + (hi - lo) * rng.random((n, 3)).astype(f32)).astype(f32)
    d = np.where(rng.random((n, 1)) < 0.7, tgt - o, rng.normal(size=(n, 3))).astype(f32)
    scale = np.where(rng.random((n, 3)) < 0.1, f32(1e-30), np.where(rng.random((n, 3)) < 0.1, f32(1e30), f32(1)))
    d = (d * scale).astype(f32)
    tmax = np.where(rng.random(n) < 0.5, np.inf, rng.uniform(0.0, 3.0, n)).astype(f32)
    accepted = check_lemma(lo, hi, plo, phi, o, d, tmax)
    assert accepted > 10_000


def ancestors_contain_vertex_boxes(flat):
    """every reference-tree box contains the vertex boxes of the triangles below it: leaves directly, interior nodes
    through their children (containment is transitive)"""
    from trace_jl_b200 import _lib as tl
    nodes, prims, v = flat.nodes, flat.prims, flat.tri_vertices
    meta = nodes["meta"].astype(np.int64)
    leaf = (meta >> 30) == 3
    off = nodes["offset"].astype(np.int64)
    li = np.nonzero(leaf)[0]
    cnt = meta[li] & 0x3FFFFFFF
    owner = np.repeat(li, cnt)
    slot = np.concatenate([np.arange(s, s + c) for s, c in zip(off[li], cnt)]) if len(li) else np.zeros(0, np.int64)
    tri = prims["kind"][slot] == tl.PRIM_TRIANGLE
    owner, slot = owner[tri], slot[tri]
    vb = v[prims["index"][slot].astype(np.int64)]
    assert np.all(nodes["bmin"][owner] <= vb.min(1)) and np.all(nodes["bmax"][owner] >= vb.max(1))
    inner = np.nonzero(~leaf)[0]
    for kid in (inner + 1, off[inner]):
        assert np.all(nodes["bmin"][inner] <= nodes["bmin"][kid]) and np.all(nodes["bmax"][inner] >= nodes["bmax"][kid])
    return len(slot)


def test_reference_tree_boxes_contain_vertex_boxes_tess_small(T):
    scene = tess_small(T)[0]
    assert ancestors_contain_vertex_boxes(scene.flatten()) > 1000


def test_reference_tree_boxes_contain_vertex_boxes_caustic(T):
    if not os.path.exists(T.scenes.ASSET_PLY):
        pytest.skip("asset missing")
    assert ancestors_contain_vertex_boxes(T.scenes.caustic_glass()[0].flatten()) > 1000
