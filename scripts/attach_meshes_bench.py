"""Several attached meshes (CompositeScene + Context.upload, trace_scene_attach_meshes_device) on the tess-1M environment
with its own sah tree: 8 UV spheres of 100 k triangles, and 64 of 10 k, at distinct positions.  Per configuration:
  replace_one_ms        one slot (3) gets a new DeviceMeshScene object of the same tensors: only that mesh is rebuilt,
                        nothing moves
  replace_one_resized_ms  slot 0 alternates between two sizes, so the kept meshes after it move (staged and rebased)
  replace_all_ms        every slot gets a new object in one call
  concat_attach_ms      today's single-mesh path: one attach of all the meshes concatenated, `with_cat` including the
                        caller's torch.cat of vertices, normals and flags, `without_cat` from arrays concatenated before
  *_phases_ms           TRACE_BVH_PROFILE=1 CUDA-event phases of the call (median of 3), and the bytes it staged for
                        kept meshes that moved
Call times are host clock around the synchronous call, median of --runs.  frame_ms (8 x 100 k only): one Whitted
frame at bench.py's tess-1M settings on the 8-slot scene against the attach of the concatenation, CUDA events over
--frames.  The GPU's name, power limit and maximum SM clock are read in the same run.  Needs a CUDA device.
usage: python scripts/attach_meshes_bench.py [--out profiles/r9_attach_meshes.json]"""
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

from bvh_build_bench import SCENES, hardware  # noqa: E402

CONFIGS = {"8x100k": (8, (224, 224)), "64x10k": (64, (71, 71))}   # UV sphere (stacks, slices): 2 slices (stacks - 1) triangles
RESIZED = {(224, 224): (212, 224), (71, 71): (67, 71)}            # slot 0's other size


def profile_line(fn):
    """one TRACE_BVH_PROFILE=1 call of fn: -> ({phase: ms}, bytes staged for kept meshes)"""
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
        line = [x for x in f.read().decode().splitlines() if x.startswith("scene attach mesh device")][-1]
    staged = re.search(r"\((\d+) bytes staged\)", line)
    return {k: float(v) for k, v in re.findall(r"([a-z-]+) ([0-9.]+) ms", line)}, int(staged.group(1)) if staged else 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(ROOT), "profiles", "r9_attach_meshes.json"))
    ap.add_argument("--runs", type=int, default=10)
    ap.add_argument("--frames", type=int, default=10)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("attach_meshes_bench.py needs a CUDA device: the attach has no CPU fallback")
    import trace_jl_b200 as T
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    result = {"hardware": hardware(), "runs": args.runs, "scene": "tess-1M", "base_builder": "sah", "mesh": "UV sphere",
              "rows": [], "not_measured": ["a base with analytic spheres or nested BVHAccels (tests cover it)",
                                           "multi-GPU attach"]}
    ms = lambda t0: 1e3 * (time.perf_counter() - t0)
    mirror = T.MirrorMaterial(T.ConstantTexture(T.RGBSpectrum(0.9)))
    kw, spp, depth = SCENES["tess-1M"]
    scene, camera, _ = T.scenes.tessellated(**kw, builder="sah")
    nb = len(scene.flatten().tri_vertices)
    H, W = camera.film.pixels.shape[:2]
    film = torch.zeros((H, W, 4), dtype=torch.float32, device="cuda:0")
    cam, fd = camera.pod(), camera.film.desc()

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        return ms(t0)

    def median_of(fn):
        every = [timed(fn) for _ in range(args.runs)]
        return statistics.median(every), every

    def profiled(fn):
        ph = [profile_line(fn) for _ in range(3)]
        return {k: statistics.median(p[0][k] for p in ph) for k in ph[0][0]}, ph[-1][1]

    def frame_ms(c):
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

    def sphere(center, stacks, slices, radius):
        v, nrm, idx = T.scenes._uv_sphere(center, radius, stacks, slices)
        tri = idx.astype(np.int64).reshape(-1, 3) - 1
        return (torch.from_numpy(v[tri]).cuda(0), torch.from_numpy(nrm[tri]).cuda(0),
                torch.full((len(tri),), 2, dtype=torch.uint8, device="cuda:0"))

    for cname, (k, (stacks, slices)) in CONFIGS.items():
        side = int(np.ceil(np.sqrt(k)))                    # a grid over x -20 .. 20, z -30 .. -10, above the heightfield
        radius = 0.45 * 20.0 / side
        centers = [(-20.0 + (j % side + 0.5) * 40.0 / side, 6.0, -30.0 + (j // side + 0.5) * 20.0 / side) for j in range(k)]
        arrays = [sphere(c, stacks, slices, radius) for c in centers]
        other = sphere(centers[0], *RESIZED[(stacks, slices)], radius)
        mk = lambda a: T.DeviceMeshScene([], a[0], [mirror], None, a[1], a[2])
        row = {"config": cname, "base_triangles": nb, "meshes": k, "mesh_triangles": [len(a[0]) for a in arrays]}
        ctx = T.Context(0, stream=stream.cuda_stream)
        ctx.upload(scene)
        meshes = [mk(a) for a in arrays]
        ctx.upload(T.CompositeScene(scene, meshes))

        def replace(j, a):
            meshes[j] = mk(a)
            ctx.upload(T.CompositeScene(scene, list(meshes)))

        row["replace_one_ms"], row["replace_one_ms_all"] = median_of(lambda: replace(3, arrays[3]))
        row["replace_one_phases_ms"], row["replace_one_staged_bytes"] = profiled(lambda: replace(3, arrays[3]))
        flip = [0]

        def resized():
            flip[0] ^= 1
            replace(0, other if flip[0] else arrays[0])

        resized()
        resized()
        row["replace_one_resized_ms"], row["replace_one_resized_ms_all"] = median_of(resized)
        row["replace_one_resized_phases_ms"], row["replace_one_resized_staged_bytes"] = profiled(resized)
        if flip[0]:
            resized()

        def replace_all():
            meshes[:] = [mk(a) for a in arrays]
            ctx.upload(T.CompositeScene(scene, list(meshes)))

        row["replace_all_ms"], row["replace_all_ms_all"] = median_of(replace_all)
        row["replace_all_phases_ms"], row["replace_all_staged_bytes"] = profiled(replace_all)
        # today's path: the concatenation attached as one mesh
        cctx = T.Context(0, stream=stream.cuda_stream)
        cctx.upload(scene)
        cat = lambda: [torch.cat([a[i] for a in arrays]) for i in range(3)]
        pre = cat()
        cctx.upload(T.CompositeScene(scene, mk(pre)))
        with_cat = lambda: cctx.upload(T.CompositeScene(scene, mk(cat())))
        without_cat = lambda: cctx.upload(T.CompositeScene(scene, mk(pre)))
        row["concat_attach_ms"] = {"with_cat": median_of(with_cat)[0], "without_cat": median_of(without_cat)[0]}
        row["concat_attach_phases_ms"] = profiled(without_cat)[0]
        if cname == "8x100k":
            replace_all()
            without_cat()
            row["frame_ms"] = {"slots": frame_ms(ctx), "concatenated": frame_ms(cctx)}
            row["spp"], row["max_depth"], row["resolution"], row["frames"] = spp, depth, list(kw["res"]), args.frames
        row["replace_one_below_concat"] = row["replace_one_ms"] < row["concat_attach_ms"]["without_cat"]
        cctx.close()
        ctx.close()
        del meshes, arrays, other, pre
        torch.cuda.empty_cache()
        print(json.dumps({k: v for k, v in row.items() if not k.endswith("_all")}), flush=True)
        result["rows"].append(row)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["hardware"]))


if __name__ == "__main__":
    main()
