"""Refit against rebuild on tess-1M and tess-10M, trees from the reference and lbvh builders (Context.refit,
trace_scene_refit[_device]).  The deformation: a heightfield wave on the ground mesh, y += A sin(1.7 x + p0) cos(1.3 z + p1)
with a seeded phase, and the mirror sphere mesh moved by A (1, 0.5, 0); A sweeps AMPLITUDES.  Per scene and builder:
  refit_device_ms   Context.refit with a CUDA tensor (the vertices never leave the GPU), host clock around the
                    synchronous call, warm, median of --runs calls with a new phase each
  refit_host_ms     the same from a numpy array (staging copy of 36 B per triangle included)
  phases_ms         TRACE_BVH_PROFILE=1 CUDA-event phases of one device and one host call (median of 3)
  rebuild_s         BVHAccel(prims, 1, builder) + Context.upload of the same deformed geometry (one call per amplitude)
  quality           per amplitude, refit tree against rebuilt tree: box tests per ray (count_nodes, a fixed seeded
                    ray set: half from the camera, half through the scene box) and, tess-1M only, one Whitted frame
                    (bench.py's settings; CUDA events over --frames frames after 2 warm-up frames)
The GPU's name, power limit and maximum SM clock are read in the same run.  Needs a CUDA device (no CPU fallback).
usage: python scripts/refit_bench.py [--out profiles/r4_refit.json] [--scenes tess-1M tess-10M]"""
import argparse
import ctypes as C
import json
import os
import re
import statistics
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(ROOT))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from bvh_build_bench import SCENES, hardware, rays  # noqa: E402

BUILDERS = ("reference", "lbvh")
AMPLITUDES = (0.0, 0.25, 1.0, 4.0)


def profiled(fn, prefix):
    """one TRACE_BVH_PROFILE=1 call of fn, the library's stderr line parsed into {phase: ms}"""
    os.environ["TRACE_BVH_PROFILE"] = "1"
    with tempfile.TemporaryFile() as f:
        sys.stderr.flush()
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["TRACE_BVH_PROFILE"]
        f.seek(0)
        line = [x for x in f.read().decode().splitlines() if x.startswith(prefix)][-1]
    return {k: float(v) for k, v in re.findall(r"([a-z-]+) ([0-9.]+) ms", line)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(ROOT), "profiles", "r4_refit.json"))
    ap.add_argument("--scenes", nargs="+", default=list(SCENES), choices=list(SCENES))
    ap.add_argument("--runs", type=int, default=20)
    ap.add_argument("--frames", type=int, default=10)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("refit_bench.py needs a CUDA device: refit has no CPU fallback")
    import trace_jl_b200 as T
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    result = {"hardware": hardware(), "runs": args.runs, "amplitudes": list(AMPLITUDES), "rows": []}
    for name in args.scenes:
        kw, spp, depth = SCENES[name]
        for builder in BUILDERS:
            ctx = T.Context(0, stream=stream.cuda_stream)          # holds the uploaded tree, refit in place
            fresh = T.Context(0, stream=stream.cuda_stream)        # uploads the rebuilt trees
            scene, camera, _ = T.scenes.tessellated(**kw, builder=builder)
            prims = [p for _, p in scene.aggregate.items]
            flat = ctx.upload(scene)
            meshes = flat.tri_sources
            n_tris = len(flat.tri_vertices)
            n_ground, n_mirror = meshes[0].n_triangles, meshes[-1].n_triangles
            base = torch.from_numpy(flat.tri_vertices).to("cuda:0")
            rng = np.random.default_rng(17)
            cam_pos = camera.camera_to_world.point([0, 0, 0]).astype(np.float32)
            ray_o, ray_d = rays(flat, cam_pos)

            def deform(a):
                p0, p1 = (float(x) for x in rng.uniform(0, 2 * np.pi, 2))
                v = base.clone()
                g = v[:n_ground]
                g[..., 1] += a * torch.sin(1.7 * g[..., 0] + p0) * torch.cos(1.3 * g[..., 2] + p1)
                v[n_tris - n_mirror:] += torch.tensor([a, 0.5 * a, 0.0], device=v.device)
                return v

            row = {"scene": name, "builder": builder, "triangles": n_tris, "nodes": int(len(flat.nodes))}
            for _ in range(3):
                ctx.refit(scene, deform(1.0))
            dev, host = [], []
            for _ in range(args.runs):
                v = deform(1.0)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ctx.refit(scene, v)
                dev.append(1e3 * (time.perf_counter() - t0))
            for _ in range(max(3, args.runs // 4)):
                v = deform(1.0).cpu().numpy()
                t0 = time.perf_counter()
                ctx.refit(scene, v)
                host.append(1e3 * (time.perf_counter() - t0))
            row["refit_device_ms"], row["refit_device_ms_all"] = statistics.median(dev), dev
            row["refit_host_ms"], row["refit_host_ms_all"] = statistics.median(host), host
            vd, vh = deform(1.0), deform(1.0).cpu().numpy()
            ph_d = [profiled(lambda: ctx.refit(scene, vd), "scene refit") for _ in range(3)]
            ph_h = [profiled(lambda: ctx.refit(scene, vh), "scene refit") for _ in range(3)]
            row["phases_ms"] = {"device": {k: statistics.median(p[k] for p in ph_d) for k in ph_d[0]},
                                "host": {k: statistics.median(p[k] for p in ph_h) for k in ph_h[0]}}
            print(json.dumps({k: v for k, v in row.items() if not k.endswith("_all")}), flush=True)

            film = cam = fd = None
            if name == "tess-1M":
                H, W = camera.film.pixels.shape[:2]
                film = torch.zeros((H, W, 4), dtype=torch.float32, device="cuda:0")
                cam, fd = camera.pod(), camera.film.desc()

            def measure(c):
                out = {}
                c.set_option("count_nodes", 1)
                c.reset_stats()
                c.intersect(ray_o, ray_d)
                out["box_tests_per_ray"] = c.stats()["nodes_visited"] / len(ray_o)
                c.set_option("count_nodes", 0)
                if film is not None:
                    def frame(i):
                        c.check(c.lib.trace_render_whitted_device(c.h, C.byref(cam), C.byref(fd), spp, depth,
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
                    out["frame_ms"] = e0.elapsed_time(e1) / args.frames
                return out

            row["quality"] = []
            for a in AMPLITUDES:
                v = deform(a)
                ctx.refit(scene, v)
                q = {"amplitude": a, "refit": measure(ctx)}
                vh = v.cpu().numpy()
                pos = 0
                for m in meshes:                                   # the same geometry on the host meshes
                    idx = m.indices.reshape(-1, 3).astype(np.int64) - 1
                    m.vertices[idx.reshape(-1)] = vh[pos:pos + m.n_triangles].reshape(-1, 3)
                    pos += m.n_triangles
                t0 = time.perf_counter()
                bvh = T.BVHAccel(prims, 1, builder=builder)
                t1 = time.perf_counter()
                fresh.upload(T.Scene(scene.lights, bvh))
                t2 = time.perf_counter()
                q["rebuild"] = {"bvhaccel_s": t1 - t0, "upload_s": t2 - t1, "total_s": t2 - t0, **measure(fresh)}
                print(json.dumps({"scene": name, "builder": builder, **q}), flush=True)
                row["quality"].append(q)
                del bvh
            row["rebuild_s"] = statistics.median(q["rebuild"]["total_s"] for q in row["quality"])
            row["rebuild_over_refit_device"] = 1e3 * row["rebuild_s"] / row["refit_device_ms"]
            if film is not None:
                row["spp"], row["max_depth"], row["resolution"], row["frames"] = spp, depth, list(kw["res"]), args.frames
            row["rays"] = len(ray_o)
            result["rows"].append(row)
            ctx.close()
            fresh.close()
            del scene, prims, flat, base, film
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["hardware"]))


if __name__ == "__main__":
    main()
