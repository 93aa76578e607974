#!/usr/bin/env python
"""hit_tree_bench.py — what the closest-hit walk on the shadow tree (option hit_tree, traverse.cuh traverse_closest_tree)
saves, per Whitted workload, with CUDA events on one GPU:
  * extend-class time per frame (k_wh_primary + k_wh_extend) with the option on and off (serial pass: lanes = 1, an
    event pair around every launch);
  * fallbacks per closest-hit ray of a frame: rays the exact check handed to the reference walk;
  * box tests and primitive tests per closest-hit ray, on random rays through trace_intersect (count_nodes 2 counts
    the walk the default path runs, count_nodes 1 the reference tree's; two box tests per pair record either way);
  * registers and spills of the closest-hit kernels, from the build's ptxas logs (when the build left them).

  python scripts/hit_tree_bench.py [--workloads tess-1M,tess-10M] [--frames 3] [--out profiles/r8_hit_tree.json]
"""
import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
CSRC = os.path.join(ROOT, "trace.jl_b200", "csrc")


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().splitlines()[0]
        return [x.strip() for x in out.split(",")]
    except Exception:
        return None


def kernel_resources():
    """{kernel signature: [registers, spill store bytes, spill load bytes]} of the slab-2 closest-hit kernels"""
    out = {}
    for f in ("api", "whitted", "sppm"):
        path = os.path.join(CSRC, f + ".ptxas.log")
        if not os.path.exists(path):
            continue
        cur, spill = None, (0, 0)
        for line in open(path):
            m = re.search(r"Compiling entry function '(\w+)'", line)
            if m:
                cur, spill = m.group(1), (0, 0)
                continue
            m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
            if m:
                spill = (int(m.group(1)), int(m.group(2)))
            m = re.search(r"Used (\d+) registers", line)
            if m and cur:
                name = subprocess.run(["c++filt"], input=cur, capture_output=True, text=True).stdout.strip()
                name = name.split("(")[0].replace("void ", "")
                if re.match(r"(k_intersect|k_wh_extend|k_wh_primary|k_sppm_cam_path|k_photon_path)<2, ", name) and \
                        ("-1" in name or "true, 0" in name):
                    out[name] = [int(m.group(1)), *spill]
                cur = None
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="tess-1M,tess-10M")
    ap.add_argument("--frames", type=int, default=3)
    ap.add_argument("--rays", type=int, default=1_000_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("hit_tree_bench.py needs a CUDA device")
    import bench
    import trace_jl_b200 as T
    from test_gpu_shadow_tree import random_rays
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    result = {"gpu": gpu_info(), "what": __doc__.strip().splitlines()[0], "kernels": kernel_resources(), "workloads": {}}
    for wl in args.workloads.split(","):
        scene, camera, spp, depth = bench.build_scene(T, wl)
        H, W = camera.film.pixels.shape[:2]
        film = torch.zeros((H, W, 4), dtype=torch.float32, device="cuda")
        cam, fd = camera.pod(), camera.film.desc()
        row = {"spp": spp, "depth": depth, "resolution": [W, H]}
        ctx = T.Context(0, stream=stream.cuda_stream)
        flat = ctx.upload(scene)
        row["shadow_tree"] = ctx.shadow_tree() is not None
        ctx.set_option("lanes", 1)

        def frame(i):
            ctx.check(ctx.lib.trace_render_whitted_device(ctx.h, C.byref(cam), C.byref(fd), spp, depth, C.c_uint64(1000 + i),
                                                          C.c_void_p(film.data_ptr())))
        for rep in range(2):                          # on, off, on, off: alternating
            for on in (1, 0):
                k = "on" if on else "off"
                ctx.set_option("hit_tree", on)
                ctx.set_option("time_kernels", 1)
                frame(0)
                torch.cuda.synchronize()
                ctx.reset_stats()
                for i in range(args.frames):
                    frame(1 + i)
                torch.cuda.synchronize()
                st = ctx.stats()
                ctx.set_option("time_kernels", 0)
                row.setdefault(f"extend_ms_per_frame_{k}_runs", []).append(st["ms_kind"][0] / args.frames)
                row[f"serial_ms_per_frame_{k}"] = sum(st["ms_kind"]) / args.frames
                row["closest_hit_rays_per_frame"] = st["rays_extend"] / args.frames
                if on:
                    row["fallbacks_per_closest_hit_ray"] = st["hit_fallbacks"] / max(1, st["rays_extend"])
        for k in ("on", "off"):
            row[f"extend_ms_per_frame_{k}"] = float(np.median(row[f"extend_ms_per_frame_{k}_runs"]))
        row["extend_ms_ratio_on_over_off"] = row["extend_ms_per_frame_on"] / row["extend_ms_per_frame_off"]
        ctx.set_option("hit_tree", 1)
        o, d, _ = random_rays(flat, args.rays, 7)
        for count, k in ((2, "on"), (1, "off")):
            ctx.set_option("count_nodes", count)
            ctx.reset_stats()
            ctx.intersect(o, d)
            st = ctx.stats()
            ctx.set_option("count_nodes", 0)
            row[f"box_tests_per_closest_hit_ray_{k}"] = st["nodes_visited"] / len(o)
            row[f"prim_tests_per_closest_hit_ray_{k}"] = st["prims_tested"] / len(o)
            if count == 2:
                row["fallbacks_per_random_ray"] = st["hit_fallbacks"] / len(o)
        result["workloads"][wl] = row
        ctx.close()
        print(json.dumps({wl: row}), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
