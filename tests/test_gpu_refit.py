"""Refit on the GPU (trace_scene_refit[_device], Context.refit): the device boxes equal the numpy restatement
(tests/test_refit_host.py) bit for bit, the refit scene answers rays exactly as a fresh upload of the same tree with
the new vertices does and renders the same images, and refused input leaves the scene untouched."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib
from test_refit_host import (boxes_equal, nested_scene, refit_flat, refit_restate, scenes_for_identity, tess_small,
                             wave)

pytestmark = pytest.mark.gpu


def same_bits(a, b):
    return np.ascontiguousarray(a).tobytes() == np.ascontiguousarray(b).tobytes()


def _caustic(T):
    if not os.path.exists(T.scenes.ASSET_PLY):
        pytest.skip("asset missing")
    return T.scenes.caustic_glass()[0]


SCENES = {
    "tess_lbvh": lambda T: tess_small(T, "lbvh")[0],
    "caustic": _caustic,
    **{k: (lambda k: lambda T: scenes_for_identity(T)[k])(k)
       for k in ("tess_reference", "tess_sah", "shadows", "shadows_mixed_leaves", "nested")},
}


def rays(flat, n, seed):
    rng = np.random.default_rng(seed)
    lo, hi = flat.nodes[0]["bmin"], flat.nodes[0]["bmax"]
    tgt = (lo + rng.random((n, 3), dtype=np.float32) * (hi - lo)).astype(np.float32)
    o = (tgt + rng.normal(size=(n, 3)).astype(np.float32) * np.float32(0.5 * np.abs(hi - lo).max())).astype(np.float32)
    d = (tgt - o).astype(np.float32)
    t_any = rng.uniform(0.2, 1.2, n).astype(np.float32)
    return o, d, t_any


def query(ctx, o, d, t_any):
    prim, t, b = ctx.intersect(o, d)
    return prim, t, b, ctx.occluded(o, d, t_any)


def assert_same_answers(a, b):
    for x, y in zip(a, b):
        assert same_bits(x, y)


@pytest.mark.parametrize("name", sorted(SCENES))
def test_refit_nodes_equal_restatement(T, ctx, name):
    scene = SCENES[name](T)
    flat = ctx.upload(scene)
    ctx.refit(scene)                                        # unchanged vertices: the uploaded boxes come back
    ident = ctx.scene_nodes()
    assert same_bits(ident, refit_restate(flat)) and boxes_equal(ident, flat.nodes)
    new = wave(flat, 0.7, seed=len(name))
    ctx.refit(scene, new)
    got = ctx.scene_nodes()
    want = refit_restate(flat, new)
    diff = np.nonzero(got.view(np.uint32).reshape(-1, 8) != want.view(np.uint32).reshape(-1, 8))[0]
    assert len(diff) == 0, f"first differing node {diff[0]}: {got[diff[0]]} vs {want[diff[0]]}"
    assert not boxes_equal(got, flat.nodes)
    ctx.refit(scene, new)                                   # deterministic
    assert same_bits(ctx.scene_nodes(), got)


@pytest.mark.parametrize("name", ("shadows", "caustic_glass", "tess_small"))
def test_identity_refit_keeps_golden_rays(T, ctx, name):
    from test_golden_rays import GOLDEN, _scene
    g = np.load(os.path.join(GOLDEN, f"rays_{name}.npz"))
    scene = _scene(T, name)
    ctx.upload(scene)
    ctx.refit(scene)
    prim, t, b = ctx.intersect(g["o"], g["d"])
    assert np.array_equal(prim, g["prim"]) and same_bits(t, g["t"]) and same_bits(b, g["b"])
    assert np.array_equal(ctx.occluded(g["o"], g["d"], g["t_max_any"]).astype(np.uint8), g["occluded"])


@pytest.mark.parametrize("name", ("tess_reference", "shadows_mixed_leaves", "nested"))
def test_deformed_hits_match_oracle_and_fresh_tree(T, ctx, name):
    scene = SCENES[name](T)
    flat = ctx.upload(scene)
    new = wave(flat, 1.5, seed=3)
    ctx.refit(scene, new)
    o, d, t_any = rays(flat, 200_000, 7)
    got = query(ctx, o, d, t_any)
    assert (got[0] != 0).mean() > 0.2
    osc = oracle_lib.OracleScene(refit_flat(flat, new))
    m = 50_000
    assert_same_answers([x[:m] for x in got[:3]], osc.intersect(o[:m], d[:m], slab=0))
    assert np.array_equal(got[3][:m], osc.occluded(o[:m], d[:m], t_any[:m], slab=0))
    if name != "tess_reference":
        return
    # a reference tree built for the deformed geometry: the same t, the primitive only differs on ties
    pos = 0
    for mesh in flat.tri_sources:
        idx = mesh.indices.reshape(-1, 3).astype(np.int64) - 1
        mesh.vertices[idx.reshape(-1)] = new[pos:pos + mesh.n_triangles].reshape(-1, 3)
        pos += mesh.n_triangles
    fresh = T.Scene(scene.lights, T.BVHAccel([p for _, p in scene.aggregate.items], 1)).flatten()
    fp, ft, _ = oracle_lib.OracleScene(fresh).intersect(o[:m], d[:m], slab=0)
    assert same_bits(ft, got[1][:m]) and (fp != got[0][:m]).mean() < 1e-3


def _whitted(ctx, camera, seed=9):
    cam, fd = camera.pod(), camera.film.desc()
    film = np.zeros_like(camera.film.pixels)
    ctx.check(ctx.lib.trace_render_whitted(ctx.h, C.byref(cam), C.byref(fd), 2, 5, C.c_uint64(seed), ctx_ptr(film)))
    return film


def _sppm(T, ctx, camera):
    cam, fd = camera.pod(), camera.film.desc()
    h, w = camera.film.pixels.shape[:2]
    rgb = np.zeros((h, w, 3), np.float32)
    ctx.check(ctx.lib.trace_render_sppm(ctx.h, C.byref(cam), C.byref(fd), 0.3, 5, 2, 20_000, 0, C.c_uint64(3),
                                        C.cast(None, T._lib.SPPM_CB),
                                        None, ctx_ptr(rgb)))
    return rgb


def same_image(a, b):
    """Equal up to the order of the film's float atomicAdd splats (two renders of one scene on one context differ
    in the last bits too); a changed tree, vertex or normal shows up far above this."""
    return np.allclose(a, b, rtol=2e-5, atol=2e-6 * float(np.abs(b).max()))


def ctx_ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _scene_scale(nodes):
    b = np.concatenate([nodes[0]["bmin"], nodes[0]["bmax"]])
    return float(np.abs(b[np.isfinite(b)]).max())


@pytest.mark.parametrize("rescale", [False, True], ids=["graph_replay", "recapture"])
def test_renders_after_refit_equal_fresh_upload(T, rescale):
    """Whitted (CUDA graph) and SPPM after a refit equal (up to splat order) the images of another context that uploaded
    the refit tree with the new vertices.  The refit context renders before the refit, so its captured graph is replayed over the new
    data when scene_scale is unchanged, and captured again when the refit scales the scene."""
    scene, camera, _ = tess_small(T)
    a, b = T.Context(0), T.Context(0)
    try:
        flat = a.upload(scene)
        before = _whitted(a, camera)
        # an asynchronous SPPM session in flight: the refit waits for it and ends it
        cam, fd = camera.pod(), camera.film.desc()
        a.check(a.lib.trace_sppm_begin(a.h, C.byref(cam), C.byref(fd), 0.3, 5, 20_000, C.c_uint64(3)))
        a.check(a.lib.trace_sppm_iterate(a.h, 1, 3))
        new = flat.tri_vertices * np.float32(1.25) if rescale else wave(flat, 0.4, seed=1)
        a.refit(scene, new)
        scale_changed = _scene_scale(a.scene_nodes()) != _scene_scale(flat.nodes)
        assert scale_changed == rescale
        film_a, rgb_a = _whitted(a, camera), _sppm(T, a, camera)
        fs = T.Scene(scene.lights, scene.aggregate)
        fs._flat = refit_flat(flat, new)
        b.upload(fs)
        film_b, rgb_b = _whitted(b, camera), _sppm(T, b, camera)
        assert same_image(film_a, film_b) and same_image(rgb_a, rgb_b)
        assert not same_image(film_a, before) and float(rgb_a.max()) > 0
    finally:
        a.close()
        b.close()


def test_degenerate_flag_follows_vertices(T):
    """Triangles shrunk until dot(g, g) underflows are degenerate after a refit and hit-testable again after the next;
    both states answer as the oracle and as a fresh upload do."""
    scene, camera, _ = tess_small(T)
    a, b = T.Context(0), T.Context(0)
    try:
        flat = a.upload(scene)
        rng = np.random.default_rng(2)
        sel = rng.choice(len(flat.tri_vertices), 2000, replace=False)
        new = flat.tri_vertices.copy()
        c = new[sel].mean(1, keepdims=True)
        new[sel] = c + (new[sel] - c) * np.float32(1e-12)
        g = np.cross(new[sel, 2] - new[sel, 0], new[sel, 1] - new[sel, 0]).astype(np.float32)
        assert ((g * g).sum(1, dtype=np.float32) == 0).all()
        o = (c[:, 0] + np.float32(3.0) * np.array([0, 1, 0], np.float32)).astype(np.float32)
        d = (c[:, 0] - o).astype(np.float32)
        t_any = np.full(len(o), 10.0, np.float32)
        for verts in (new, flat.tri_vertices):
            a.refit(scene, verts)
            fs = T.Scene(scene.lights, scene.aggregate)
            fs._flat = refit_flat(flat, verts)
            b.upload(fs)
            got = query(a, o, d, t_any)
            assert_same_answers(got, query(b, o, d, t_any))
            osc = oracle_lib.OracleScene(fs._flat)
            assert_same_answers(got[:3], osc.intersect(o, d, slab=0))
            assert np.array_equal(got[3], osc.occluded(o, d, t_any, slab=0))
    finally:
        a.close()
        b.close()


def test_new_normals_change_shading_like_a_fresh_upload(T):
    scene, camera, _ = tess_small(T)
    a, b = T.Context(0), T.Context(0)
    try:
        flat = a.upload(scene)
        before = _whitted(a, camera)
        rng = np.random.default_rng(4)
        nrm = (flat.tri_normals + rng.normal(size=flat.tri_normals.shape) * 0.2).astype(np.float32)
        nrm /= np.linalg.norm(nrm, axis=-1, keepdims=True).astype(np.float32)
        a.refit(scene, flat.tri_vertices, nrm)
        film = _whitted(a, camera)
        fs = T.Scene(scene.lights, scene.aggregate)
        fs._flat = refit_flat(flat, flat.tri_vertices, nrm)
        b.upload(fs)
        assert same_image(film, _whitted(b, camera)) and not same_image(film, before)
        a.refit(scene, flat.tri_vertices)                   # normals=None keeps the new ones
        assert same_image(_whitted(a, camera), film)
    finally:
        a.close()
        b.close()


def test_torch_tensor_path_equals_numpy_path(T, ctx):
    torch = pytest.importorskip("torch")
    scene = nested_scene(T)
    flat = ctx.upload(scene)
    new = wave(flat, 0.9, seed=8)
    o, d, t_any = rays(flat, 50_000, 3)
    ctx.refit(scene, new)
    want_nodes, want = ctx.scene_nodes(), query(ctx, o, d, t_any)
    ctx.refit(scene, flat.tri_vertices)
    ctx.refit(scene, torch.from_numpy(new).to(f"cuda:{ctx.device}"))
    assert same_bits(ctx.scene_nodes(), want_nodes)
    assert_same_answers(query(ctx, o, d, t_any), want)
    with pytest.raises(ValueError):
        ctx.refit(scene, torch.from_numpy(new).to(f"cuda:{ctx.device}").double())


def test_refused_input_leaves_scene_untouched(T):
    c, other = T.Context(0), T.Context(0)
    try:
        lib = c.lib
        assert lib.trace_scene_refit(c.h, 0, None, None, 0, None) != 0
        assert b"no scene" in lib.trace_last_error(c.h)
        scene = T.scenes.shadows(resolution=32)[0]
        flat = c.upload(scene)
        o, d, t_any = rays(flat, 20_000, 1)
        nodes0, ans0 = c.scene_nodes(), query(c, o, d, t_any)
        sb = np.ascontiguousarray(flat.sphere_bounds)
        v = np.ascontiguousarray(wave(flat, 0.3))
        n = len(v)
        bad = v.copy()
        bad[n // 2, 1, 2] = np.nan
        nan_n = flat.tri_normals.copy()
        nan_n[0, 0, 0] = np.nan
        cases = [  # (message, n_tris, vertices, normals, n_spheres, sphere bounds)
            (b"NaN", n, bad, None, len(sb), sb),
            (b"NaN", n, v, nan_n, len(sb), sb),
            (b"triangles given", n - 1, v, None, len(sb), sb),
            (b"no sphere bounds", n, v, None, 0, None),
        ]
        for msg, nt, vv, nn, ns, sbb in cases:
            rc = lib.trace_scene_refit(c.h, nt, ctx_ptr(vv), None if nn is None else ctx_ptr(nn), ns,
                                       None if sbb is None else ctx_ptr(sbb))
            assert rc != 0 and msg in lib.trace_last_error(c.h), msg
            assert same_bits(c.scene_nodes(), nodes0)
            assert_same_answers(query(c, o, d, t_any), ans0)
        with pytest.raises(RuntimeError, match="NaN"):
            c.refit(scene, bad)
        assert not flat.stale
        with pytest.raises(ValueError, match="not the one uploaded"):
            c.refit(T.scenes.shadows(resolution=32)[0])
        c.refit(scene, v)
        assert flat.stale
        with pytest.raises(RuntimeError, match="stale"):
            other.upload(scene)
    finally:
        c.close()
        other.close()
