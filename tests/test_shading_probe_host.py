"""CPU side of the call-by-call shading checks: the device probe compiles for sm_100a with the library's flags, the
numpy restatement of add_sample! equals the oracle's bit for bit, and the oracle's batched entry points equal its
single calls."""
import ctypes as C

import numpy as np

import oracle_lib
import probe_lib
import shading_cases as sc
from trace_jl_b200 import _lib as tl


def test_probe_compiles_with_the_makefile_flags(tmp_path):
    flags = probe_lib.makefile_nvccflags()
    for f in ("-fmad=false", "arch=compute_100a,code=sm_100a", "-O3"):
        assert any(f in x for x in flags), f
    assert "-ffp-contract=off" in " ".join(flags)
    so = probe_lib.build(str(tmp_path))
    syms = C.CDLL(so)      # resolves against libtrace_cuda.so (ctx_pack_materials); no device needed to load
    for name in ("probe_pack_materials", "probe_bsdf_f", "probe_bsdf_sample", "probe_hit_record", "probe_radical_inverse",
                 "probe_rng"):
        assert hasattr(syms, name)


def _film_desc(rng, radius, crop):
    import trace_jl_b200 as T
    film = T.Film([64, 48], T.Bounds2(crop[:2], crop[2:]), T.LanczosSincFilter(radius, 3.0), 1.0, 1.0, None)
    return film.desc()


def test_add_sample_restatement_equals_oracle():
    """Random positions, radii, tile bounds and crops, tiles clipped at pixel 1 included: the same touched pixels and
    the same weights as ref_film_tile_add_sample, bit for bit."""
    rng = np.random.default_rng(3)
    L = oracle_lib.lib()
    radii = [(0.5, 0.5), (1, 1), (1.5, 1.5), (2, 2), (2, 1), (2.5, 2.5), (4, 4), (4, 1.5), (0.7, 3.3)]
    crops = [(0, 0, 1, 1), (0.25, 0.125, 0.75, 0.9), (0.0, 0.5, 0.3, 1.0)]
    calls = 0
    for radius in radii:
        for crop in crops:
            fd = _film_desc(rng, radius, crop)
            sx0, sy0, sx1, sy1 = sc.sample_bounds(fd)
            for _ in range(40):
                bx0 = int(rng.integers(sx0, sx1 + 1)) // 16 * 16 if rng.random() < 0.5 else int(rng.integers(sx0, sx1 + 1))
                by0 = int(rng.integers(sy0, sy1 + 1))
                bx1, by1 = min(bx0 + 15, sx1), min(by0 + 15, sy1)
                tb = sc.tile_bounds(fd, np.array([bx0]), np.array([by0]), np.array([bx1]), np.array([by1]))
                tb = tuple(int(t[0]) for t in tb)
                tw, th = tb[2] - tb[0] + 1, tb[3] - tb[1] + 1
                if tw <= 0 or th <= 0:
                    continue
                fx = np.float32(bx0 + rng.uniform(0, bx1 - bx0 + 1))
                fy = np.float32(by0 + rng.uniform(0, by1 - by0 + 1))
                if rng.random() < 0.1:
                    fx = np.float32(np.floor(fx)) + np.float32(0.5)          # on a pixel centre: table column 1
                contrib = np.zeros((th, tw, 3), np.float32)
                wsum = np.zeros((th, tw), np.float32)
                rgb = np.array([np.nan, 1, 1], np.float32)                    # NaN marks every touched pixel
                tbv = np.array(tb, np.int32)
                L.ref_film_tile_add_sample(C.byref(fd), oracle_lib.p(tbv), C.c_float(fx), C.c_float(fy), oracle_lib.p(rgb),
                                           oracle_lib.p(contrib), oracle_lib.p(wsum))
                want = np.zeros((th, tw), np.float32)
                touched = np.zeros((th, tw), bool)
                tba = tuple(np.array([t]) for t in tb)
                for _, x, y, w in sc.add_sample_footprint(fd, tba, np.array([fx]), np.array([fy])):
                    want[y - tb[1], x - tb[0]] += w
                    touched[y - tb[1], x - tb[0]] = True
                assert np.array_equal(np.isnan(contrib[..., 0]), touched), (radius, crop, tb, fx, fy)
                assert np.array_equal(wsum.view(np.uint32), want.view(np.uint32)), (radius, crop, tb, fx, fy)
                calls += 1
    assert calls > 800


def test_rng_restatement_equals_oracle():
    rng = np.random.default_rng(4)
    seed = rng.integers(0, 2**63, 2000, dtype=np.uint64)
    abc = rng.integers(0, 2**32, (2000, 3), dtype=np.uint64)
    got = sc.rng_uniform(seed, abc[:, 0], abc[:, 1], abc[:, 2])
    L = oracle_lib.lib()
    want = np.array([L.ref_rng(int(s), int(a), int(b), int(c)) for s, (a, b, c) in zip(seed, abc)], np.float32)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_batched_bsdf_entry_points_equal_single_calls():
    rng = np.random.default_rng(5)
    mats = sc.materials()
    wo, wi = sc.bsdf_f_inputs(rng, 200)
    sel = rng.integers(0, len(wo), 3000)
    wo, wi = wo[sel], wi[sel]
    q = np.stack([rng.integers(0, len(mats), len(wo)), rng.integers(0, 2, len(wo)),
                  rng.choice(sc.F_FLAGS, len(wo))], 1).astype(np.int32)
    f, nl = oracle_lib.bsdf_f_batch(mats, q, wo, wi)
    u = sc.sample_u(rng, len(wo))[: len(wo)]
    qs = q.copy()
    qs[:, 2] = rng.choice(sc.S_TYPES, len(wo))
    s, snl = oracle_lib.bsdf_sample_batch(mats, qs, wo, u)
    L = oracle_lib.lib()
    for i in range(len(wo)):
        one = np.zeros(3, np.float32)
        n = L.ref_bsdf_f(mats[q[i, 0]:].ctypes.data_as(C.c_void_p), int(q[i, 1]), oracle_lib.p(wo[i]), oracle_lib.p(wi[i]),
                         int(q[i, 2]), oracle_lib.p(one))
        assert n == nl[i] and np.array_equal(one.view(np.uint32), f[i].view(np.uint32)), i
        out = np.zeros(8, np.float32)
        n = L.ref_bsdf_sample(mats[qs[i, 0]:].ctypes.data_as(C.c_void_p), int(qs[i, 1]), oracle_lib.p(wo[i]),
                              oracle_lib.p(u[i]), int(qs[i, 2]), oracle_lib.p(out))
        assert n == snl[i] and np.array_equal(out.view(np.uint32), s[i].view(np.uint32)), i
    assert set(nl.tolist()) >= {0, 1, 2}


def test_batched_hit_records_equal_single_calls():
    import trace_jl_b200 as T
    scene, camera, _ = T.scenes.shadows(resolution=32)
    osc = oracle_lib.OracleScene(scene.flatten())
    rng = np.random.default_rng(6)
    o = np.tile(np.array([[0.4, 1.5, 1.0]], np.float32), (500, 1))
    tgt = np.stack([rng.uniform(-1, 2, 500), rng.uniform(-0.5, 1, 500), rng.uniform(-4, -1, 500)], 1).astype(np.float32)
    d = (tgt - o).astype(np.float32)
    batch = osc.hit_records(o, d)
    for i in range(len(o)):
        one = np.zeros(24, np.float32)
        oracle_lib.lib().ref_hit_record(osc.h, oracle_lib.p(o[i]), oracle_lib.p(d[i]), C.c_float(np.inf), oracle_lib.p(one))
        assert np.array_equal(one.view(np.uint32), batch[i].view(np.uint32)), i
    assert 0 < np.count_nonzero(batch[:, 0]) < len(o)
