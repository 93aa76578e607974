"""ctypes binding of the CPU oracle (oracle/libtrace_ref.so).  TEST INFRASTRUCTURE: imported only from tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs."""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
LIB = os.path.join(ORACLE_DIR, "libtrace_ref.so")

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB):
            subprocess.check_call(["make", "libtrace_ref.so"], cwd=ORACLE_DIR)
        L = C.CDLL(LIB)
        P = C.c_void_p
        L.ref_bvh_build.restype = C.c_int
        L.ref_bvh_build.argtypes = [P, C.c_int64, C.c_int, C.POINTER(P)]
        L.ref_bvh_num_nodes.restype = C.c_int64
        L.ref_bvh_num_nodes.argtypes = [P]
        L.ref_bvh_max_depth.restype = C.c_int
        L.ref_bvh_max_depth.argtypes = [P]
        L.ref_bvh_copy.argtypes = [P, P, P]
        L.ref_bvh_free.argtypes = [P]
        L.ref_scene_create.restype = P
        L.ref_scene_create.argtypes = [P]
        L.ref_scene_free.argtypes = [P]
        L.ref_intersect.argtypes = [P, P, P, P, C.c_int64, P, P, C.c_int, P, C.c_int]
        L.ref_occluded.argtypes = [P, P, P, P, C.c_int64, P, C.c_int, P, C.c_int]
        L.ref_hit_record.argtypes = [P, P, P, C.c_float, P]
        L.ref_prim_hit_record.argtypes = [P, C.c_int64, P, P, C.c_float, P]
        L.ref_render_whitted.argtypes = [P, P, P, C.c_int, C.c_int, C.c_uint64, P, C.c_int, C.c_int64, P]
        L.ref_render_whitted_tiles.argtypes = [P, P, P, C.c_int, C.c_int, C.c_uint64, P, P, C.c_int64, C.c_int, P]
        L.ref_render_sppm.argtypes = [P, P, P, C.c_float, C.c_int, C.c_int, C.c_int64, C.c_uint64, P, C.c_int, P]
        L.ref_bounds_intersect.argtypes = [P, P, P, P, C.c_float, C.POINTER(C.c_float), C.POINTER(C.c_float)]
        L.ref_bounds_intersect_p.argtypes = [P, P, P, P, C.c_float, C.c_int]
        L.ref_fresnel_dielectric.restype = C.c_float
        L.ref_fresnel_dielectric.argtypes = [C.c_float, C.c_float, C.c_float]
        L.ref_fresnel_specular_sample.argtypes = [P, P, C.c_float, C.c_float, P, P, P]
        L.ref_microfacet_reflection_sample.argtypes = [P, C.c_float, C.c_float, C.c_int, C.c_float, C.c_float, P, P, P]
        L.ref_microfacet_transmission_sample.argtypes = [P, C.c_float, C.c_float, C.c_float, C.c_float, P, P, P]
        L.ref_lanczos.restype = C.c_float
        L.ref_lanczos.argtypes = [C.c_float] * 5
        L.ref_radical_inverse.restype = C.c_float
        L.ref_radical_inverse.argtypes = [C.c_int64, C.c_uint64]
        L.ref_roughness_to_alpha.restype = C.c_float
        L.ref_roughness_to_alpha.argtypes = [C.c_float]
        L.ref_bsdf_f.argtypes = [P, C.c_int, P, P, C.c_int, P]
        L.ref_bsdf_sample.argtypes = [P, C.c_int, P, P, C.c_int, P]
        L.ref_bsdf_f_batch.argtypes = [P, C.c_int64, P, P, P, P, P]
        L.ref_bsdf_sample_batch.argtypes = [P, C.c_int64, P, P, P, P, P]
        L.ref_hit_record_batch.argtypes = [P, C.c_int64, P, P, P, P, C.c_int]
        L.ref_film_tile_add_sample.argtypes = [P, P, C.c_float, C.c_float, P, P, P]
        L.ref_rng.restype = C.c_float
        L.ref_rng.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32]
        _lib = L
    return _lib


def p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def f3(x):
    return np.ascontiguousarray(x, dtype=np.float32)


def bvh_build(bounds, max_node_prims=1):
    """-> (nodes structured array, order, max_depth)"""
    from trace_jl_b200 import _lib as tl
    L = lib()
    bounds = np.ascontiguousarray(bounds, dtype=np.float32)
    h = C.c_void_p()
    rc = L.ref_bvh_build(p(bounds), len(bounds), max_node_prims, C.byref(h))
    assert rc == 0, rc
    nodes = np.zeros(L.ref_bvh_num_nodes(h), dtype=tl.node_dtype)
    order = np.zeros(len(bounds), dtype=np.uint32)
    L.ref_bvh_copy(h, p(nodes), p(order))
    depth = L.ref_bvh_max_depth(h)
    L.ref_bvh_free(h)
    return nodes, order, depth


def bsdf_f_batch(mats, q, wo, wi):
    """ref_bsdf_f over n inputs; q: [n, 3] (material index, mode, flags) -> f [n, 3], lobe count [n]"""
    mats = np.ascontiguousarray(mats)
    q = np.ascontiguousarray(q, dtype=np.int32)
    wo, wi = f3(wo), f3(wi)
    f, nl = np.zeros((len(q), 3), np.float32), np.zeros(len(q), np.int32)
    lib().ref_bsdf_f_batch(p(mats), len(q), p(q), p(wo), p(wi), p(f), p(nl))
    return f, nl


def bsdf_sample_batch(mats, q, wo, u):
    """ref_bsdf_sample over n inputs; q: [n, 3] (material index, mode, type) -> [n, 8] (wi, f, pdf, type), lobe count [n]"""
    mats = np.ascontiguousarray(mats)
    q = np.ascontiguousarray(q, dtype=np.int32)
    wo, u = f3(wo), f3(u)
    out, nl = np.zeros((len(q), 8), np.float32), np.zeros(len(q), np.int32)
    lib().ref_bsdf_sample_batch(p(mats), len(q), p(q), p(wo), p(u), p(out), p(nl))
    return out, nl


class OracleScene:
    def __init__(self, flat):
        self.flat = flat
        d = flat.desc()
        self.h = lib().ref_scene_create(C.byref(d))
        self.threads = os.cpu_count() or 1

    def __del__(self):
        try:
            if self.h:
                lib().ref_scene_free(self.h)
                self.h = None
        except Exception:
            pass

    def intersect(self, o, d, t_max=None, slab=0, counters=False):
        o = f3(o).reshape(-1, 3)
        d = f3(d).reshape(-1, 3)
        n = len(o)
        t = np.full(n, np.inf, np.float32) if t_max is None else f3(t_max).copy()
        prim = np.zeros(n, np.uint32)
        b = np.zeros((n, 2), np.float32)
        cnt = np.zeros(3, np.uint64)
        lib().ref_intersect(self.h, p(o), p(d), p(t), n, p(prim), p(b), slab, p(cnt) if counters else None, self.threads)
        return (prim, t, b, cnt) if counters else (prim, t, b)

    def occluded(self, o, d, t_max=None, slab=0):
        o = f3(o).reshape(-1, 3)
        d = f3(d).reshape(-1, 3)
        n = len(o)
        t = np.full(n, np.inf, np.float32) if t_max is None else f3(t_max)
        out = np.zeros(n, np.uint8)
        lib().ref_occluded(self.h, p(o), p(d), p(t), n, p(out), slab, None, self.threads)
        return out.astype(bool)

    def hit_record(self, o, d, t_max=np.inf, prim=-1):
        """prim = -1: intersect!(bvh, ray); prim >= 0: intersect(shape, ray) on that BVH-ordered primitive alone"""
        out = np.zeros(24, np.float32)
        o, d = f3(o), f3(d)
        lib().ref_prim_hit_record(self.h, prim, p(o), p(d), C.c_float(t_max), p(out))
        if out[0] == 0:
            return None
        return dict(t=out[1], p=out[2:5], ng=out[5:8], ns=out[8:11], ss=out[11:14], ts=out[14:17], wo=out[17:20],
                    uv=out[20:22], prim=int(out[22]), material=int(out[23]))

    def hit_records(self, o, d, t_max=None):
        """ref_hit_record over n rays -> float32 [n, 24] (hit, t, p, ng, ns, ss, ts, wo, uv, original, material)"""
        o, d = f3(o).reshape(-1, 3), f3(d).reshape(-1, 3)
        t = None if t_max is None else f3(t_max)
        out = np.zeros((len(o), 24), np.float32)
        lib().ref_hit_record_batch(self.h, len(o), p(o), p(d), p(t), p(out), self.threads)
        return out

    def render_whitted(self, cam, fd, spp, max_depth, seed, film_xyzw, max_tiles=0, threads=None):
        cnt = np.zeros(2, np.uint64)
        rc = lib().ref_render_whitted(self.h, C.byref(cam), C.byref(fd), spp, max_depth, C.c_uint64(seed), p(film_xyzw),
                                      threads or self.threads, max_tiles, p(cnt))
        assert rc == 0
        return cnt

    def render_whitted_tiles(self, cam, fd, spp, max_depth, seed, film_xyzw, tiles, threads=None):
        """Only the 16x16 sample tiles in `tiles` (k = ty * n_tiles_x + tx), e.g. one rank's share k % world == rank."""
        cnt = np.zeros(2, np.uint64)
        tl = np.ascontiguousarray(tiles, dtype=np.int64)
        rc = lib().ref_render_whitted_tiles(self.h, C.byref(cam), C.byref(fd), spp, max_depth, C.c_uint64(seed), p(film_xyzw),
                                            p(tl), len(tl), threads or self.threads, p(cnt))
        assert rc == 0
        return cnt

    def render_sppm(self, cam, fd, r0, max_depth, n_iter, photons, seed, rgb, threads=None):
        cnt = np.zeros(2, np.uint64)
        rc = lib().ref_render_sppm(self.h, C.byref(cam), C.byref(fd), C.c_float(r0), max_depth, n_iter, photons,
                                   C.c_uint64(seed), p(rgb), threads or self.threads, p(cnt))
        assert rc == 0
        return cnt
