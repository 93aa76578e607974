"""The device's shading functions held call by call against the CPU oracle (-m gpu): bsdf_f, bsdf_sample, the hit
record, the Halton radical inverse and the counter-based RNG, each run through tests/cuda/shading_probe.cu on the
library's own headers and compared with the oracle's unit entry points on the same inputs.

Equal means bit-equal, except that NaN equals NaN whatever its payload (the device's canonical NaN and x86's differ
in sign).  Where a device libm function feeds a result the comparison is bounded, and the function is named:

- bsdf_sample, diffuse lobes: concentric_disk calls cosf / sinf (CUDA: at most 2 ULP; glibc: under 1 ULP), so
  wi.x and wi.y may differ by a few ULP of 1 and wi.z = sqrt(1 - x^2 - y^2) inherits an absolute error in wi.z^2.
- bsdf_sample, microfacet lobes with the scaled wo within tr_sample11's `cth > 0.9999` branch: double cos / sin (both
  sides under 1 ULP in double) rounded to float: the slope differs by at most 1 float ULP, then moves wh and wi.
- hit records on spheres: theta = acosf(z / r) and sinf(theta) (CUDA: 2 ULP each) feed dpdv, so ng, ns and ts.

Bounds (the tests print the measured maxima per class):
- diffuse and near-normal microfacet samples: |d wi.x|, |d wi.y| <= 2e-6, a few ULP of 1 from the cos / sin
  difference with a wide margin; |d (wi.z^2)| <= 4e-6, since wi.z^2 = 1 - x^2 - y^2 inherits 2 (|x| + |y|) times
  the x, y error and wi.z itself is ill-conditioned at the horizon; f, pdf and f |cos| / pdf within a relative 1e-3
  where |wi.z| >= 1e-3 on both sides (a few ULP of direction, amplified by the lobes' condition number, which grows
  as alpha falls to its 1e-3 clamp).  A "none" sample (pdf 0) on one side only is allowed where the other side drew
  a diffuse direction with wi.z^2 <= 8 * 2^-24, and such samples are counted: u0 or u1 at 0 or 1 put the disk
  point on the unit circle, so 1 - x^2 - y^2 is only cosf / sinf rounding, and wi.z = sqrt(max(0, ...)) is 0 on
  one side and up to sqrt(8 * 2^-24) = 6.9e-4 on the other (a pdf of 0 there makes the sample "none").
- sphere hit records: p, wo, ss bit-equal; ng, ns, ts within 4e-6 per component (2 ULP in acosf and sinf move the
  unnormalised dpdv by a few ULP of the radius).
"""
import numpy as np
import pytest

import oracle_lib
import probe_lib
import shading_cases as sc
from trace_jl_b200 import _lib as tl

pytestmark = pytest.mark.gpu


def same_bits(a, b):
    """element-wise: bit-equal, or both NaN"""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


def report(label, ok, dev=0.0):
    print(f"{label}: {ok.size} calls, {int(np.count_nonzero(ok))} bit-equal, largest deviation {dev:.3g}")


@pytest.fixture(scope="module")
def mats():
    return sc.materials()


# ---------------------------------------------------------------- bsdf_f
def test_bsdf_f_bit_for_bit(ctx, mats):
    """Every material, mode 0 and 1, every flag set, on the edge direction sets and uniform pairs: no device libm on
    this path (pow4 goes through double on both sides, the roughness remap's logf runs on the host), so bit for bit."""
    rng = np.random.default_rng(21)
    wo, wi = sc.bsdf_f_inputs(rng, 20000)
    sub = rng.integers(0, len(wo), 3000)
    qs, wos, wis = [], [], []
    for m in range(len(mats)):
        for mode in (0, 1):
            for flags in sc.F_FLAGS:
                idx = np.arange(len(wo)) if flags == sc.LB_ALL else sub
                qs.append(np.tile(np.int32([m, mode, flags]), (len(idx), 1)))
                wos.append(wo[idx]); wis.append(wi[idx])
    q, wo, wi = np.concatenate(qs), np.concatenate(wos), np.concatenate(wis)
    f, nl = probe_lib.bsdf_f(ctx, mats, q, wo, wi)
    rf, rnl = oracle_lib.bsdf_f_batch(mats, q, wo, wi)
    assert np.array_equal(nl, rnl), "lobe counts differ"
    assert set(nl.tolist()) == {0, 1, 2}
    ok = same_bits(f, rf).all(axis=1)
    report("bsdf_f", ok)
    bad = np.flatnonzero(~ok)
    assert len(bad) == 0, f"{len(bad)} of {len(q)} bsdf_f calls differ; first: q {q[bad[0]]} wo {wo[bad[0]]} wi {wi[bad[0]]} " \
                          f"gpu {f[bad[0]]} oracle {rf[bad[0]]}"
    assert np.count_nonzero(f) > len(f) // 4


# ---------------------------------------------------------------- bsdf_sample
def _sample_inputs(rng, mats):
    e = sc.edge_directions(rng)
    uni = sc._unit(rng.normal(size=(2000, 3)))
    # within tr_sample11's near-normal branch for every alpha: cos theta > 1 - 1e-9 before the alpha scaling
    th = rng.uniform(0, 3e-5, 200)
    ph = rng.uniform(0, 2 * np.pi, 200)
    nn = np.stack([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th)], 1).astype(np.float32)
    nn = np.concatenate([nn, nn * np.float32([1, 1, -1])]).astype(np.float32)
    wo_pool = np.concatenate([e, uni, nn]).astype(np.float32)
    u_pool = sc.sample_u(rng, 2000)
    n_edge_u = len(u_pool) - 2000
    half = int(np.flatnonzero((u_pool == np.float32(0.5)).all(axis=1))[0])
    qs, wos, us = [], [], []
    for m in range(len(mats)):
        for mode in (0, 1):
            for typ in sc.S_TYPES:
                k = 6000
                wi_idx = rng.integers(0, len(wo_pool), k)
                u_idx = np.where(rng.random(k) < 0.5, rng.integers(0, n_edge_u, k), rng.integers(0, len(u_pool), k))
                # every edge direction with u = (0.5, 0.5) and with an edge u
                wi_idx = np.concatenate([wi_idx, np.arange(len(e)), np.arange(len(e))])
                u_idx = np.concatenate([u_idx, np.full(len(e), half), rng.integers(0, n_edge_u, len(e))])
                qs.append(np.tile(np.int32([m, mode, typ]), (len(wi_idx), 1)))
                wos.append(wo_pool[wi_idx]); us.append(u_pool[u_idx])
    return np.concatenate(qs), np.concatenate(wos), np.concatenate(us)


def near_normal_branch(packed, q, out_type, wo):
    """microfacet samples whose scaled wo takes tr_sample11's `cth > 0.9999` branch (float32, as tr_sample_wh)"""
    f = np.float32
    m = packed[q[:, 0]]
    ax = m["alpha_u"].astype(f)
    ay = np.where(m["kind"] == tl.MAT_PLASTIC, m["alpha_u"], m["alpha_v"]).astype(f)
    w = np.where((wo[:, 2] < 0)[:, None], -wo, wo).astype(f)
    x, y, z = w[:, 0] * ax, w[:, 1] * ay, w[:, 2]
    with np.errstate(divide="ignore", invalid="ignore"):
        cth = (f(1) / np.sqrt((x * x + y * y) + z * z)) * z
    glossy = (out_type.astype(np.int64) & sc.LB_GLOSSY) != 0
    return glossy & (cth > f(0.9999))


def test_bsdf_sample_against_oracle(ctx, mats):
    """Same materials, types LB_ALL, specular only and non-specular; u0 = k / mc exactly, u = 0.5, 0, 1 - 2^-24; wo
    within the near-normal branch.  Specular lobes and microfacet samples off that branch: all outputs bit-equal.  The
    sampled type: equal everywhere.  Diffuse and near-normal microfacet samples: the bounds of the module docstring."""
    rng = np.random.default_rng(22)
    q, wo, u = _sample_inputs(rng, mats)
    packed = probe_lib.pack_materials(ctx, mats)
    g, nl = probe_lib.bsdf_sample(ctx, mats, q, wo, u)
    r, rnl = oracle_lib.bsdf_sample_batch(mats, q, wo, u)
    assert np.array_equal(nl, rnl)
    gt, rt = g[:, 7], r[:, 7]
    none_g, none_r = g[:, 6] == 0, r[:, 6] == 0
    one_sided = none_g != none_r
    # a "none" on one side only: the other side drew a diffuse direction whose disk point lies on the unit circle up
    # to the cosf / sinf rounding, i.e. wi.z^2 = 1 - x^2 - y^2 within 8 ULP of 1 from 0
    other_z2 = np.where(none_g, r[:, 2], g[:, 2]).astype(np.float64) ** 2
    other_diffuse = (np.where(none_g, rt, gt).astype(np.int64) & sc.LB_DIFFUSE) != 0
    horizon = other_diffuse & (other_z2 <= 8 * 2.0 ** -24)
    off = np.flatnonzero(one_sided & ~horizon)
    assert len(off) == 0, f"{len(off)} one-sided 'none' samples off the horizon; first: q {q[off[0]]} wo {wo[off[0]]} " \
                          f"u {u[off[0]]} gpu {g[off[0]]} oracle {r[off[0]]}"
    both = ~one_sided
    assert np.array_equal(gt[both], rt[both]), f"sampled type differs on {np.count_nonzero(gt[both] != rt[both])} samples"
    typ = np.where(none_g, rt, gt).astype(np.int64)
    diffuse = (typ & sc.LB_DIFFUSE) != 0
    libm = diffuse | near_normal_branch(packed, q, typ, wo)
    exact = both & ~libm
    ok = same_bits(g[exact], r[exact]).all(axis=1)
    report("bsdf_sample exact (specular, microfacet off the near-normal branch)", ok)
    bad = np.flatnonzero(exact)[~ok]
    assert len(bad) == 0, f"{len(bad)} samples differ; first: q {q[bad[0]]} wo {wo[bad[0]]} u {u[bad[0]]} gpu {g[bad[0]]} oracle {r[bad[0]]}"
    assert np.count_nonzero(exact & (typ >= sc.LB_SPECULAR)) > 1000 and np.count_nonzero(exact & ((typ & sc.LB_GLOSSY) != 0)) > 1000
    # bounded classes
    for label, sel in (("diffuse (cosf / sinf)", both & diffuse), ("microfacet near-normal (double cos / sin)", both & libm & ~diffuse)):
        a, b = g[sel].astype(np.float64), r[sel].astype(np.float64)
        same = same_bits(g[sel], r[sel])                  # per output; equal values (NaN or Inf included) deviate by 0
        eq = same.all(axis=1)
        away = (np.abs(a[:, 2]) >= 1e-3) & (np.abs(b[:, 2]) >= 1e-3) & (a[:, 6] > 0) & (b[:, 6] > 0)
        with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
            def dev(x, y, s):                              # a NaN here (one side only) fails the bounds below
                return np.where(s, 0.0, np.abs(x - y)).max(initial=0.0)

            def rel(x, y, s):
                return np.where(s, 0.0, np.abs(x - y) / np.maximum(np.maximum(np.abs(x), np.abs(y)), 1e-30)).max(initial=0.0)
            wa = a[:, 3:6] * np.abs(a[:, 2:3]) / a[:, 6:7]
            wb = b[:, 3:6] * np.abs(b[:, 2:3]) / b[:, 6:7]
            dxy = dev(a[:, :2], b[:, :2], same[:, :2])
            dz2 = dev(a[:, 2] ** 2, b[:, 2] ** 2, same[:, 2])
            rf = rel(a[away, 3:6], b[away, 3:6], same[away, 3:6])
            rp = rel(a[away, 6], b[away, 6], same[away, 6])
            rw = rel(wa[away], wb[away], same[away, 2:7].all(axis=1)[:, None])
        report(f"bsdf_sample {label}", eq, max(dxy, dz2, rf, rp, rw))
        print(f"  |d wi.xy| {dxy:.3g}  |d wi.z^2| {dz2:.3g}  rel f {rf:.3g}  rel pdf {rp:.3g}  rel f|cos|/pdf {rw:.3g}  "
              f"({np.count_nonzero(away)} away from the horizon)")
        assert dxy <= 2e-6 and dz2 <= 4e-6, label
        assert rf <= 1e-3 and rp <= 1e-3 and rw <= 1e-3, label
    print(f"bsdf_sample one-sided 'none' at the horizon: {np.count_nonzero(one_sided)} of {len(q)}, "
          f"largest other-side wi.z^2 {other_z2[one_sided].max(initial=0.0):.3g}")


# ---------------------------------------------------------------- hit records
def _hit_record_check(T, ctx, scene, o, d, label, tmax=None):
    flat = ctx.upload(scene)
    osc = oracle_lib.OracleScene(flat)
    o, d = np.ascontiguousarray(o, np.float32), np.ascontiguousarray(d, np.float32)
    prim, t, b = ctx.intersect(o, d, tmax)
    rec = osc.hit_records(o, d, tmax)
    original = flat.prims["original"]
    assert len(np.unique(original)) == len(original)
    slot_of = np.empty(int(original.max()) + 1, np.int64)
    slot_of[original] = np.arange(len(original))
    # rays whose closest hit is already bit-equal (primitive and t)
    hit = (prim != 0) & (rec[:, 0] == 1) & (rec[:, 22] == (prim.astype(np.float64) - 1)) & same_bits(rec[:, 1], t)
    assert np.count_nonzero(hit) > 0.3 * len(o) and np.count_nonzero((prim != 0) & ~hit) == 0, label
    slot = slot_of[prim[hit].astype(np.int64) - 1]
    out, ids = probe_lib.hit_record(ctx, slot, o[hit], d[hit], b[hit])
    r = rec[hit]
    assert np.array_equal(ids[:, 0].astype(np.float32), r[:, 23]) and np.array_equal(ids[:, 1].astype(np.float32), r[:, 22]), label
    sphere = flat.prims["kind"][slot] == tl.PRIM_SPHERE
    names = ["p", "ng", "ns", "ss", "ts", "wo"]
    for k, name in enumerate(names):
        g, w = out[:, 3 * k:3 * k + 3], r[:, 2 + 3 * k:5 + 3 * k]
        eq = same_bits(g, w).all(axis=1)
        tri_bad = np.flatnonzero(~eq & ~sphere)
        assert len(tri_bad) == 0, f"{label}: triangle {name} differs on {len(tri_bad)} hits; first gpu {g[tri_bad[0]]} oracle {w[tri_bad[0]]}"
        if sphere.any():
            dev = float(np.abs(g[sphere].astype(np.float64) - w[sphere]).max())
            report(f"hit record {label} sphere {name}", eq[sphere], dev)
            if name in ("p", "wo", "ss"):
                assert eq[sphere].all(), f"{label}: sphere {name} not bit-equal ({dev})"
            else:
                assert dev <= 4e-6, f"{label}: sphere {name} off by {dev}"
    report(f"hit record {label} triangles", np.ones(np.count_nonzero(~sphere), bool))
    return flat


def test_hit_records(T, ctx):
    import test_gpu_parity as gp
    scenes = [("tess-small",) + T.scenes.tessellated(cells=48, stacks=26, slices=24, res=(160, 90))[:2]]
    import os
    if os.path.exists(T.scenes.ASSET_PLY):
        scenes.append(("caustic-mesh",) + T.scenes.caustic_glass(resolution=64)[:2])
    mat = T.MatteMaterial(T.ConstantTexture(T.RGBSpectrum(0.5)), T.ConstantTexture(0.0))
    prims = [T.GeometricPrimitive(T.Sphere(T.ShapeCore(T.translate([0, 0, 0]), False), 1.0, -0.5, 0.7, 300.0), mat),
             T.GeometricPrimitive(T.Sphere(T.ShapeCore(T.translate([3, 0, 0]), True), 1.2, 360.0), mat),
             T.GeometricPrimitive(T.Sphere(T.ShapeCore(T.translate([0, 3, 0]) * T.scale(1, -1, 1), False), 0.8, -0.8, 0.3, 200.0), mat)]
    # reverse orientation with and without vertex normals (TRACE_TRI_FLIP), and a triangle whose vertex normals are
    # parallel to p1 - p0, so ns x ss vanishes and build_interaction takes coordinate_system
    prims += [T.GeometricPrimitive(t, mat) for t in T.create_triangle_mesh(
        T.ShapeCore(T.translate([-3, 0, 0]), True), 2, [1, 2, 3, 1, 3, 4], 4, [[0, 0, 0], [1, 0, 0], [1, 1, 0.5], [0, 1, 0]])]
    prims += [T.GeometricPrimitive(t, mat) for t in T.create_triangle_mesh(
        T.ShapeCore(T.translate([-3, -3, 0]), True), 2, [1, 2, 3, 1, 3, 4], 4, [[0, 0, 0], [1, 0, 0], [1, 1, 0.5], [0, 1, 0]],
        [[0.1, 0.2, 1], [0, 0, 1], [0.2, 0, 1], [0, 0.3, 1]])]
    prims += [T.GeometricPrimitive(t, mat) for t in T.create_triangle_mesh(
        T.ShapeCore(T.translate([3, -3, 0]), False), 1, [1, 2, 3], 3, [[0, 0, 0], [1, 0, 0], [0, 1, 0]],
        [[1, 0, 0], [1, 0, 0], [1, 0, 0]])]
    scene = T.Scene([T.PointLight(T.translate([0, 5, 5]), T.RGBSpectrum(10.0))], T.BVHAccel(prims))
    film = T.Film([64, 64], T.Bounds2([0, 0], [1, 1]), T.LanczosSincFilter([1, 1], 3.0), 1.0, 1.0, None)
    cam = T.PerspectiveCamera(T.look_at([0, 0, 12], [0, 0, 0]), T.Bounds2([-3000, -3000], [3000, 3000]), 0, 1, 0, 1e6, 90.0, film)
    scenes.append(("spheres+flipped", scene, cam))
    for label, scn, camera in scenes:
        sets = gp.ray_sets(T, scn, camera, 60000, 5)
        o = np.concatenate([v[0] for v in sets.values()])
        d = np.concatenate([v[1] for v in sets.values()])
        if label == "spheres+flipped":          # aimed at the hand-made triangles, too
            tgt = np.concatenate([np.random.default_rng(1).uniform([-3, -3, 0], [-2, -2, 0.5], (20000, 3)),
                                  np.random.default_rng(2).uniform([-3, 0, 0], [-2, 1, 0.5], (20000, 3)),
                                  np.random.default_rng(3).uniform([3, -3, 0], [3.5, -2.5, 0], (20000, 3))]).astype(np.float32)
            oo = np.tile(np.float32([[0.2, 0.1, 6]]), (len(tgt), 1))
            o = np.concatenate([o, oo]); d = np.concatenate([d, (tgt - oo).astype(np.float32)])
        _hit_record_check(T, ctx, scn, o, d, label)


# ---------------------------------------------------------------- Halton and RNG
def test_radical_inverse_bit_for_bit():
    rng = np.random.default_rng(23)
    primes = [2] + [p for p in range(3, 8200) if all(p % k for k in range(2, int(p ** 0.5) + 1))][:1023]
    bi, av = [], []
    for base_index in range(1024):
        base = primes[base_index]
        a = [0, 1, 2**32 - 1, 2**32, 2**32 + 1, 2**53 - 1]
        k, v = 1, base
        while v < 2**62:
            a += [v - 1, v, v + 1]
            k, v = k + 1, v * base
        a += rng.integers(0, 2**62, 16, dtype=np.uint64).tolist() + rng.integers(0, 4096, 8).tolist()
        bi += [base_index] * len(a)
        av += a
    bi, av = np.array(bi, np.int32), np.array(av, np.uint64)
    g = probe_lib.radical_inverse(bi, av)
    L = oracle_lib.lib()
    r = np.array([L.ref_radical_inverse(int(b), int(a)) for b, a in zip(bi, av)], np.float32)
    ok = same_bits(g, r)
    report("radical_inverse", ok)
    assert ok.all(), f"{np.count_nonzero(~ok)} differ; first base index {bi[~ok][0]} a {av[~ok][0]}"


def test_rng_bit_for_bit():
    rng = np.random.default_rng(24)
    n = 1_000_000
    seed = rng.integers(0, 2**64 - 1, n, dtype=np.uint64, endpoint=True)
    abc = rng.integers(0, 2**32, (n, 3), dtype=np.uint64).astype(np.uint32)
    g = probe_lib.rng(seed, abc)
    want = sc.rng_uniform(seed, abc[:, 0], abc[:, 1], abc[:, 2])       # pinned to ref_rng in test_shading_probe_host.py
    L = oracle_lib.lib()
    direct = np.array([L.ref_rng(int(seed[i]), int(abc[i, 0]), int(abc[i, 1]), int(abc[i, 2])) for i in range(5000)], np.float32)
    assert np.array_equal(direct.view(np.uint32), want[:5000].view(np.uint32))
    ok = same_bits(g, want)
    report("rng_uniform", ok)
    assert ok.all()
