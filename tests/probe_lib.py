"""ctypes binding of tests/cuda/shading_probe.cu, the device half of the call-by-call shading checks.  TEST
INFRASTRUCTURE: the probe is built once per process into a temporary directory with the NVCCFLAGS of
trace.jl_b200/csrc/Makefile (so -fmad=false and the other flags cannot drift from the library's) and linked against
libtrace_cuda.so."""
import ctypes as C
import os
import re
import shutil
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "trace.jl_b200", "csrc")
SOURCE = os.path.join(ROOT, "tests", "cuda", "shading_probe.cu")
NVCC = "/usr/local/cuda/bin/nvcc"

_lib = None
_dir = None


def makefile_nvccflags():
    """NVCCFLAGS of the library's Makefile with $(ARCH) expanded, $(EXTRA) dropped and -Xptxas -v kept."""
    text = open(os.path.join(CSRC, "Makefile")).read()
    var = dict(re.findall(r"^(\w+)\s*\??=\s*(.*)$", text, re.M))
    flags = var["NVCCFLAGS"].replace("$(ARCH)", var["ARCH"]).replace("$(EXTRA)", "")
    return flags.split()


def build(out_dir):
    """nvcc <Makefile flags> -shared shading_probe.cu -ltrace_cuda -> out_dir/libshading_probe.so; returns its path."""
    so = os.path.join(out_dir, "libshading_probe.so")
    cmd = [NVCC, *makefile_nvccflags(), "-shared", SOURCE, "-o", so, "-L" + CSRC, "-ltrace_cuda",
           "-Xlinker", "-rpath=" + CSRC]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("shading probe build failed:\n" + r.stdout[-4000:])
    return so


def lib():
    global _lib, _dir
    if _lib is None:
        from trace_jl_b200 import _lib as tl
        tl.load()                                   # libtrace_cuda.so first: the probe resolves its symbols there
        _dir = tempfile.mkdtemp(prefix="shading_probe_")
        try:
            L = C.CDLL(build(_dir))
        finally:
            shutil.rmtree(_dir, ignore_errors=True)     # the loaded library stays mapped
        P = C.c_void_p
        L.probe_pack_materials.argtypes = [P, C.c_int64, P, P]
        L.probe_bsdf_f.argtypes = [P, C.c_int64, P, C.c_int64, P, P, P, P, P]
        L.probe_bsdf_sample.argtypes = [P, C.c_int64, P, C.c_int64, P, P, P, P, P]
        L.probe_hit_record.argtypes = [P, C.c_int64, P, P, P, P, P, P]
        L.probe_radical_inverse.argtypes = [C.c_int64, P, P, P]
        L.probe_rng.argtypes = [C.c_int64, P, P, P]
        _lib = L
    return _lib


# DeviceMaterial (device_common.cuh)
device_material_dtype = np.dtype([("kind", "<u4"), ("a", "<f4", 3), ("b", "<f4", 3), ("eta", "<f4"), ("alpha_u", "<f4"),
                                  ("alpha_v", "<f4"), ("specular", "<u4"), ("pad", "<u4")])


def p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _check(rc, what):
    if rc != 0:
        raise RuntimeError(f"{what} failed ({rc})")


def pack_materials(ctx, mats):
    out = np.zeros(len(mats), device_material_dtype)
    _check(lib().probe_pack_materials(ctx.h, len(mats), p(mats), p(out)), "probe_pack_materials")
    return out


def bsdf_f(ctx, mats, q, wo, wi):
    """q: int32 [n, 3] (material, mode, flags) -> f float32 [n, 3], lobe count int32 [n]"""
    q, wo, wi = (np.ascontiguousarray(x) for x in (q.astype(np.int32), wo.astype(np.float32), wi.astype(np.float32)))
    n = len(q)
    f, nl = np.zeros((n, 3), np.float32), np.zeros(n, np.int32)
    _check(lib().probe_bsdf_f(ctx.h, len(mats), p(mats), n, p(q), p(wo), p(wi), p(f), p(nl)), "probe_bsdf_f")
    return f, nl


def bsdf_sample(ctx, mats, q, wo, u):
    """q: int32 [n, 3] (material, mode, type) -> float32 [n, 8] (wi, f, pdf, sampled type), lobe count int32 [n]"""
    q, wo, u = (np.ascontiguousarray(x) for x in (q.astype(np.int32), wo.astype(np.float32), u.astype(np.float32)))
    n = len(q)
    out, nl = np.zeros((n, 8), np.float32), np.zeros(n, np.int32)
    _check(lib().probe_bsdf_sample(ctx.h, len(mats), p(mats), n, p(q), p(wo), p(u), p(out), p(nl)), "probe_bsdf_sample")
    return out, nl


def hit_record(ctx, slot, o, d, b):
    """-> float32 [n, 18] (p, ng, ns, ss, ts, wo), uint32 [n, 2] (material, original)"""
    slot = np.ascontiguousarray(slot, dtype=np.uint32)
    o, d, b = (np.ascontiguousarray(x, dtype=np.float32) for x in (o, d, b))
    n = len(slot)
    out, ids = np.zeros((n, 18), np.float32), np.zeros((n, 2), np.uint32)
    _check(lib().probe_hit_record(ctx.h, n, p(slot), p(o), p(d), p(b), p(out), p(ids)), "probe_hit_record")
    return out, ids


def radical_inverse(base_index, a):
    base_index = np.ascontiguousarray(base_index, dtype=np.int32)
    a = np.ascontiguousarray(a, dtype=np.uint64)
    out = np.zeros(len(a), np.float32)
    _check(lib().probe_radical_inverse(len(a), p(base_index), p(a), p(out)), "probe_radical_inverse")
    return out


def rng(seed, abc):
    seed = np.ascontiguousarray(seed, dtype=np.uint64)
    abc = np.ascontiguousarray(abc, dtype=np.uint32)
    out = np.zeros(len(seed), np.float32)
    _check(lib().probe_rng(len(seed), p(seed), p(abc), p(out)), "probe_rng")
    return out
