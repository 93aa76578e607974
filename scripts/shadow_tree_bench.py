#!/usr/bin/env python
"""shadow_tree_bench.py — what the shadow tree (option shadow_tree, traverse.cuh traverse_shadow) costs and saves, per
Whitted workload, with CUDA events on one GPU:
  * k_wh_shadow time per frame with the option on and off (serial pass: lanes = 1, an event pair around every launch);
  * fallback rate: shadow rays of a frame that the exact check handed to the reference walk;
  * box tests per shadow ray, on surface-to-light rays through trace_occluded (option count_nodes; the reference walk
    counts one box per node step, the shadow walk two per pair record);
  * extra upload time (upload with the option on minus off) and extra device memory (64 B per pair record);
  * refit time with and without the shadow tree (trace_scene_refit_device, same vertices).

  python scripts/shadow_tree_bench.py [--workloads tess-1M,tess-10M] [--frames 3] [--out profiles/r5_shadow_tree.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().splitlines()[0]
        return [x.strip() for x in out.split(",")]
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="tess-1M,tess-10M")
    ap.add_argument("--frames", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("shadow_tree_bench.py needs a CUDA device")
    import bench
    import trace_jl_b200 as T
    from test_gpu_shadow_tree import shadow_rays
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    result = {"gpu": gpu_info(), "what": __doc__.strip().splitlines()[0], "workloads": {}}
    for wl in args.workloads.split(","):
        scene, camera, spp, depth = bench.build_scene(T, wl)
        H, W = camera.film.pixels.shape[:2]
        film = torch.zeros((H, W, 4), dtype=torch.float32, device="cuda")
        cam, fd = camera.pod(), camera.film.desc()
        row = {"spp": spp, "depth": depth, "resolution": [W, H]}
        ctxs = {}
        for on in (0, 1):
            ctx = T.Context(0, stream=stream.cuda_stream)
            ctx.set_option("shadow_tree", on)
            ctx.upload(scene)                         # first upload: allocations
            walls = []
            for _ in range(5):
                ctx._scene = None
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ctx.upload(scene)
                torch.cuda.synchronize()
                walls.append((time.perf_counter() - t0) * 1e3)
            row[f"upload_ms_{'on' if on else 'off'}"] = float(np.median(walls))
            row[f"upload_ms_all_{'on' if on else 'off'}"] = [round(w, 2) for w in walls]
            ctxs[on] = ctx
        n_pairs = ctxs[1].shadow_tree().shape[0] if ctxs[1].shadow_tree() is not None else 0
        row["shadow_tree_pairs"] = n_pairs
        row["extra_device_bytes"] = 64 * n_pairs
        row["extra_upload_ms"] = row["upload_ms_on"] - row["upload_ms_off"]
        for on, ctx in ctxs.items():
            ctx.set_option("lanes", 1)
            ctx.set_option("time_kernels", 1)

            def frame(i):
                ctx.check(ctx.lib.trace_render_whitted_device(ctx.h, C.byref(cam), C.byref(fd), spp, depth, C.c_uint64(1000 + i),
                                                              C.c_void_p(film.data_ptr())))
            frame(0)
            torch.cuda.synchronize()
            ctx.reset_stats()
            for i in range(args.frames):
                frame(1 + i)
            torch.cuda.synchronize()
            st = ctx.stats()
            k = f"{'on' if on else 'off'}"
            row[f"shadow_ms_per_frame_{k}"] = st["ms_kind"][1] / args.frames
            row[f"extend_ms_per_frame_{k}"] = st["ms_kind"][0] / args.frames
            row[f"serial_ms_per_frame_{k}"] = sum(st["ms_kind"]) / args.frames
            row[f"shadow_rays_per_frame"] = st["rays_shadow"] / args.frames
            if on:
                row["fallback_rate"] = st["shadow_fallbacks"] / max(1, st["rays_shadow"])
            ctx.set_option("time_kernels", 0)
        flat = scene.flatten()
        o, d, t = shadow_rays(ctxs[1], flat, 1_000_000, 7)
        for on, ctx in ctxs.items():
            ctx.set_option("count_nodes", 1)
            ctx.reset_stats()
            ctx.occluded(o, d, t)
            st = ctx.stats()
            ctx.set_option("count_nodes", 0)
            row[f"box_tests_per_shadow_ray_{'on' if on else 'off'}"] = st["nodes_visited"] / len(o)
            row[f"prim_tests_per_shadow_ray_{'on' if on else 'off'}"] = st["prims_tested"] / len(o)
        verts = torch.from_numpy(np.ascontiguousarray(flat.gather_vertices(), np.float32)).cuda()
        for on, ctx in ctxs.items():
            ctx.refit(scene, verts)                   # first refit: topology
            walls = []
            for _ in range(5):
                t0 = time.perf_counter()
                ctx.refit(scene, verts)
                walls.append((time.perf_counter() - t0) * 1e3)
            row[f"refit_ms_{'on' if on else 'off'}"] = float(np.median(walls))
            flat.stale = False
        row["shadow_ms_ratio_on_over_off"] = row["shadow_ms_per_frame_on"] / row["shadow_ms_per_frame_off"]
        result["workloads"][wl] = row
        for ctx in ctxs.values():
            ctx.close()
        print(json.dumps({wl: row}), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
