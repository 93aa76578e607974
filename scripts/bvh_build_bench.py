"""Tree builders side by side: the host reference build, the host SAH build and the GPU LBVH build (trace_bvh_build,
trace_bvh_build_sah, trace_bvh_build_gpu) on tess-1M and tess-10M.  Per builder and scene:
  build_s      wall time of the library call (the GPU call is synchronous: both copies included), one warm-up, median of 5
  phases_ms    lbvh only: the TRACE_BVH_PROFILE=1 CUDA-event phases of the call, median of 3 profiled calls
  upload_s     wall time of Context.upload (host packing of the flat scene + trace_scene_upload), one fresh scene
  box_tests_per_ray   count_nodes over a fixed seeded set of rays (half from the camera, half through the scene box)
  frame_ms     tess-1M only: one Whitted frame (bench.py's tess-1M settings, default options), CUDA events over 20 frames
               after 2 warm-up frames
The GPU's name, power limit and maximum SM clock are read in the same run.  Needs a CUDA device (no CPU fallback).
usage: python scripts/bvh_build_bench.py [--out profiles/r3_bvh_build.json] [--scenes tess-1M tess-10M]"""
import argparse
import ctypes as C
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

SCENES = {   # bench.py's WORKLOADS: scene kwargs, spp, depth
    "tess-1M": (dict(cells=600, stacks=266, slices=264, res=(1920, 1080), window=((-50.0, -28.125), (50.0, 28.125))), 16, 5),
    "tess-10M": (dict(cells=1900, stacks=835, slices=834, res=(4096, 4096), window=((-50.0, -50.0), (50.0, 50.0))), 64, 8),
}
BUILDERS = ("reference", "sah", "lbvh")


def lib_build(lib, tl, builder, bounds, m=1):
    h = C.c_void_p()
    t0 = time.perf_counter()
    if builder == "lbvh":
        rc = lib.trace_bvh_build_gpu(0, tl.ptr(bounds), len(bounds), m, C.byref(h))
    else:
        fn = lib.trace_bvh_build if builder == "reference" else lib.trace_bvh_build_sah
        rc = fn(tl.ptr(bounds), len(bounds), m, C.byref(h))
    dt = time.perf_counter() - t0
    if rc != 0:
        raise RuntimeError(f"{builder} build failed ({rc})")
    lib.trace_bvh_free(h)
    return dt


def profiled_phases(lib, tl, bounds):
    """one TRACE_BVH_PROFILE=1 call of the GPU build, its stderr line parsed into {phase: ms}"""
    os.environ["TRACE_BVH_PROFILE"] = "1"
    with tempfile.TemporaryFile() as f:
        sys.stderr.flush()
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            lib_build(lib, tl, "lbvh", bounds)
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["TRACE_BVH_PROFILE"]
        f.seek(0)
        line = [x for x in f.read().decode().splitlines() if x.startswith("bvh build gpu")][-1]
    return {k: float(v) for k, v in re.findall(r"([a-z-]+) ([0-9.]+) ms", line)}


def tree_depth(nodes):
    level, depth = np.zeros(1, np.int64), 0
    while len(level):
        depth += 1
        inner = level[(nodes["meta"][level] >> 30) != 3]
        level = np.concatenate([inner + 1, nodes["offset"][inner].astype(np.int64)])
    return depth


def rays(flat, camera_pos, n=2_000_000, seed=5):
    rng = np.random.default_rng(seed)
    lo, hi = flat.nodes[0]["bmin"], flat.nodes[0]["bmax"]
    target = (lo + rng.random((n, 3), dtype=np.float32) * (hi - lo)).astype(np.float32)
    origin = np.where(rng.random((n, 1)) < 0.5, camera_pos[None].astype(np.float32),
                      target + rng.normal(size=(n, 3)).astype(np.float32) * np.float32(0.05 * np.linalg.norm(hi - lo)))
    return origin.astype(np.float32), (target - origin).astype(np.float32)


def hardware():
    import torch
    out = {"gpu": torch.cuda.get_device_name(0), "host_cpus": os.cpu_count()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        out["power_limit_w"], out["sm_max_mhz"] = float(q[0]), float(q[1])
    except Exception as e:                                    # (reported, not fatal: the times stand without it)
        out["power_limit_w"] = f"not read: {e}"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_bvh_build.json"))
    ap.add_argument("--scenes", nargs="+", default=list(SCENES), choices=list(SCENES))
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--frames", type=int, default=20)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bvh_build_bench.py needs a CUDA device: the GPU builder has no CPU fallback")
    import trace_jl_b200 as T
    from trace_jl_b200 import _lib as tl
    lib = tl.load()
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = T.Context(0, stream=stream.cuda_stream)
    result = {"hardware": hardware(), "runs": args.runs, "rows": []}
    for name in args.scenes:
        kw, spp, depth = SCENES[name]
        scene, camera, _ = T.scenes.tessellated(**kw, builder="lbvh")
        prims = [p for _, p in scene.aggregate.items]
        bounds = scene.aggregate.prim_bounds
        cam_pos = camera.camera_to_world.point([0, 0, 0]).astype(np.float32)
        ray_o = ray_d = None
        for builder in BUILDERS:
            row = {"scene": name, "builder": builder, "primitives": int(len(bounds))}
            lib_build(lib, tl, builder, bounds)                                   # warm-up
            times = [lib_build(lib, tl, builder, bounds) for _ in range(args.runs)]
            row["build_s"] = statistics.median(times)
            row["build_s_all"] = times
            if builder == "lbvh":
                ph = [profiled_phases(lib, tl, bounds) for _ in range(3)]
                row["phases_ms"] = {k: statistics.median(p[k] for p in ph) for k in ph[0]}
            t0 = time.perf_counter()
            bvh = T.BVHAccel(prims, 1, builder=builder)
            row["bvhaccel_s"] = time.perf_counter() - t0
            row["nodes"], row["depth"] = int(len(bvh.nodes)), tree_depth(bvh.nodes)
            sc = T.Scene(scene.lights, bvh)
            t0 = time.perf_counter()
            flat = ctx.upload(sc)
            row["upload_s"] = time.perf_counter() - t0
            if ray_o is None:
                ray_o, ray_d = rays(flat, cam_pos)
            ctx.set_option("count_nodes", 1)
            ctx.reset_stats()
            ctx.intersect(ray_o, ray_d)
            row["box_tests_per_ray"] = ctx.stats()["nodes_visited"] / len(ray_o)
            row["rays"] = len(ray_o)
            ctx.set_option("count_nodes", 0)
            if name == "tess-1M":
                H, W = camera.film.pixels.shape[:2]
                film = torch.zeros((H, W, 4), dtype=torch.float32, device="cuda:0")
                cam, fd = camera.pod(), camera.film.desc()

                def frame(i):
                    ctx.check(ctx.lib.trace_render_whitted_device(ctx.h, C.byref(cam), C.byref(fd), spp, depth,
                                                                  C.c_uint64(1000 + i), C.c_void_p(film.data_ptr())))
                for i in range(2):
                    frame(i)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for i in range(args.frames):
                    frame(2 + i)
                e1.record(stream)
                torch.cuda.synchronize()
                row["frame_ms"] = e0.elapsed_time(e1) / args.frames
                row["frames"] = args.frames
                row["spp"], row["max_depth"], row["resolution"] = spp, depth, list(kw["res"])
            print(json.dumps(row), flush=True)
            result["rows"].append(row)
            del bvh, sc, flat
        del scene, prims, bounds
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["hardware"]))


if __name__ == "__main__":
    main()
