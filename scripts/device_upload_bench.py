"""The device mesh upload (DeviceMeshScene + Context.upload, trace_scene_upload_mesh_device) against the host path it
replaces (BVHAccel(builder="lbvh") + Context.upload) on tess-1M and tess-10M.  Per scene:
  host_path_s       BVHAccel(prims, 1, builder="lbvh") and Context.upload of the same triangles, host clock, median
                    of --host-runs
  device_first_ms   upload of a DeviceMeshScene of CUDA tensors into a fresh context (its grow-only buffers empty)
  device_warm_ms    the same into a warm context, a new DeviceMeshScene object per call, median of --runs
  scene_ctor_ms     DeviceMeshScene(...) of CUDA tensors (checks and the exact device bound), median of --runs
  numpy_ms          DeviceMeshScene(...) of numpy arrays (the move to the device included) + upload, median of 3
  phases_ms         TRACE_BVH_PROFILE=1 CUDA-event phases of warm device uploads (median of 3)
  same_tree         the device path's nodes equal the host path's (boxes float ==, structure words identical)
  frame_ms          tess-1M: one Whitted frame (bench.py's settings) on either path's scene, CUDA events over --frames
  sweep             the refit bench's wave amplitudes: a device rebuild (new DeviceMeshScene + upload) against
                    Context.refit of the scene uploaded undeformed; call time (host clock around the synchronous call,
                    median of 5) and, tess-1M, the frame time after each
The GPU's name, power limit and maximum SM clock are read in the same run.  Needs a CUDA device (no CPU fallback).
usage: python scripts/device_upload_bench.py [--out profiles/r6_device_upload.json] [--scenes tess-1M tess-10M]"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(ROOT))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from bvh_build_bench import SCENES, hardware  # noqa: E402
from refit_bench import AMPLITUDES, profiled  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(ROOT), "profiles", "r6_device_upload.json"))
    ap.add_argument("--scenes", nargs="+", default=list(SCENES), choices=list(SCENES))
    ap.add_argument("--runs", type=int, default=10)
    ap.add_argument("--host-runs", type=int, default=2)
    ap.add_argument("--frames", type=int, default=10)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("device_upload_bench.py needs a CUDA device: the device upload has no CPU fallback")
    import trace_jl_b200 as T
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    result = {"hardware": hardware(), "runs": args.runs, "amplitudes": list(AMPLITUDES), "rows": []}
    ms = lambda t0: 1e3 * (time.perf_counter() - t0)
    for name in args.scenes:
        kw, spp, depth = SCENES[name]
        scene, camera, _ = T.scenes.tessellated(**kw, builder="lbvh")
        prims = [p for _, p in scene.aggregate.items]
        flat = scene.flatten()
        n = len(flat.tri_vertices)
        ids = np.zeros(n, np.int32)
        ids[flat.prims["index"].astype(np.int64)] = flat.prims["material"]
        host_arrays = (flat.tri_vertices, flat.tri_normals, flat.tri_flags, ids)
        dev = [torch.from_numpy(np.ascontiguousarray(a)).cuda(0) for a in host_arrays]
        n_ground, n_mirror = flat.tri_sources[0].n_triangles, flat.tri_sources[-1].n_triangles
        row = {"scene": name, "triangles": n}

        def mk(v=None):
            return T.DeviceMeshScene(scene.lights, dev[0] if v is None else v, flat.materials, dev[3], dev[1], dev[2])

        # host path
        hctx = T.Context(0, stream=stream.cuda_stream)
        host = []
        for _ in range(args.host_runs):
            t0 = time.perf_counter()
            hs = T.Scene(scene.lights, T.BVHAccel(prims, 1, builder="lbvh"))
            t1 = time.perf_counter()
            hctx.upload(hs)
            host.append({"bvhaccel_s": t1 - t0, "upload_s": time.perf_counter() - t1})
        row["host_path_s"] = {k: statistics.median(h[k] for h in host) for k in host[0]}
        row["host_path_s"]["total"] = row["host_path_s"]["bvhaccel_s"] + row["host_path_s"]["upload_s"]
        # device path
        dctx = T.Context(0, stream=stream.cuda_stream)
        ds = mk()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dctx.upload(ds)
        row["device_first_ms"] = ms(t0)
        warm, ctor = [], []
        for _ in range(args.runs):
            t0 = time.perf_counter()
            ds = mk()
            ctor.append(ms(t0))
            t0 = time.perf_counter()
            dctx.upload(ds)
            warm.append(ms(t0))
        row["device_warm_ms"], row["device_warm_ms_all"] = statistics.median(warm), warm
        row["scene_ctor_ms"] = statistics.median(ctor)
        npt = []
        for _ in range(3):
            t0 = time.perf_counter()
            dctx.upload(T.DeviceMeshScene(scene.lights, host_arrays[0], flat.materials, host_arrays[3], host_arrays[1],
                                          host_arrays[2]))
            npt.append(ms(t0))
        row["numpy_ms"] = statistics.median(npt)
        ph = [profiled(lambda: dctx.upload(mk()), "scene upload mesh device") for _ in range(3)]
        row["phases_ms"] = {k: statistics.median(p[k] for p in ph) for k in ph[0]}
        dctx.upload(ds)
        a, b = dctx.scene_nodes(), hctx.scene_nodes()
        row["nodes"] = len(a)
        row["same_tree"] = bool(len(a) == len(b) and np.array_equal(a["bmin"], b["bmin"]) and np.array_equal(a["bmax"], b["bmax"])
                                and np.array_equal(a["offset"], b["offset"]) and np.array_equal(a["meta"], b["meta"]))
        print(json.dumps({k: v for k, v in row.items() if not k.endswith("_all")}), flush=True)

        film = cam = fd = None
        if name == "tess-1M":
            H, W = camera.film.pixels.shape[:2]
            film = torch.zeros((H, W, 4), dtype=torch.float32, device="cuda:0")
            cam, fd = camera.pod(), camera.film.desc()

        def frame_ms(c):
            if film is None:
                return None

            def frame(i):
                c.check(c.lib.trace_render_whitted_device(c.h, C.byref(cam), C.byref(fd), spp, depth, C.c_uint64(1000 + i),
                                                          C.c_void_p(film.data_ptr())))
            for i in range(2):
                frame(i)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for i in range(args.frames):
                frame(2 + i)
            e1.record(stream)
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / args.frames

        if film is not None:
            row["frame_ms"] = {"host_path": frame_ms(hctx), "device_path": frame_ms(dctx)}
            row["spp"], row["max_depth"], row["resolution"], row["frames"] = spp, depth, list(kw["res"]), args.frames
        hctx.close()
        del hs, hctx
        # rebuild against refit over the wave sweep (the refit bench's deformation)
        rctx = T.Context(0, stream=stream.cuda_stream)
        base = dev[0]
        rs = mk()
        rctx.upload(rs)
        rng = np.random.default_rng(17)

        def deform(amp):
            p0, p1 = (float(x) for x in rng.uniform(0, 2 * np.pi, 2))
            v = base.clone()
            g = v[:n_ground]
            g[..., 1] += amp * torch.sin(1.7 * g[..., 0] + p0) * torch.cos(1.3 * g[..., 2] + p1)
            v[n - n_mirror:] += torch.tensor([amp, 0.5 * amp, 0.0], device=v.device)
            return v

        row["sweep"] = []
        for amp in AMPLITUDES:
            v = deform(amp)
            q = {"amplitude": amp}
            for kind in ("refit", "rebuild"):
                times = []
                for _ in range(5):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    if kind == "refit":
                        rctx.refit(rs, v)
                    else:
                        dctx.upload(mk(v))
                    times.append(ms(t0))
                q[kind] = {"call_ms": statistics.median(times), "frame_ms": frame_ms(rctx if kind == "refit" else dctx)}
            print(json.dumps({"scene": name, **q}), flush=True)
            row["sweep"].append(q)
        result["rows"].append(row)
        rctx.close()
        dctx.close()
        del scene, prims, flat, dev, base, film, ds, rs
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["hardware"]))


if __name__ == "__main__":
    main()
