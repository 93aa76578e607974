"""The mesh attach (CompositeScene + Context.upload, trace_scene_attach_mesh_device): a UV-sphere mesh of 10 k, 100 k
and 1 M triangles attached to a tess-1M and a tess-10M environment with its own sah tree, against the two ways of
putting the same geometry on the GPU without it.  Per (base, mesh):
  first_attach_ms   the first attach after the environment's upload (it moves the base's records up one slot)
  attach_ms         later attaches, a new DeviceMeshScene object of the same tensors per call, median of --runs
  phases_ms         TRACE_BVH_PROFILE=1 CUDA-event phases of a later attach (median of 3)
  device_upload_ms  the environment's and the mesh's triangles as one DeviceMeshScene (all rebuilt), median of --runs
  host_path_s       BVHAccel(environment items + mesh, 1, builder="lbvh") and Context.upload, host clock, one run
All call times are host clock around the synchronous call.  frame_ms, tess-1M with the 100 k mesh: one Whitted frame
(bench.py's settings) on the composed scene against the all-LBVH device upload of the same triangles, CUDA events over
--frames.  The GPU's name, power limit and maximum SM clock are read in the same run.  Needs a CUDA device.
usage: python scripts/attach_mesh_bench.py [--out profiles/r7_attach_mesh.json] [--scenes tess-1M tess-10M]"""
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
from refit_bench import profiled  # noqa: E402

MESHES = {"10k": (71, 71), "100k": (224, 224), "1M": (708, 707)}   # UV sphere (stacks, slices): 2 slices (stacks - 1) triangles
CENTER, RADIUS = (0.0, 6.0, -20.0), 3.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(ROOT), "profiles", "r7_attach_mesh.json"))
    ap.add_argument("--scenes", nargs="+", default=list(SCENES), choices=list(SCENES))
    ap.add_argument("--runs", type=int, default=10)
    ap.add_argument("--frames", type=int, default=10)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("attach_mesh_bench.py needs a CUDA device: the attach has no CPU fallback")
    import trace_jl_b200 as T
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    result = {"hardware": hardware(), "runs": args.runs, "base_builder": "sah", "mesh": "UV sphere", "rows": [],
              "not_measured": ["attach of a mesh to a base with analytic spheres or nested BVHAccels (tests cover it)",
                               "multi-GPU attach"]}
    ms = lambda t0: 1e3 * (time.perf_counter() - t0)
    ident = T.ShapeCore(T.Transformation(), False)
    mirror = T.MirrorMaterial(T.ConstantTexture(T.RGBSpectrum(0.9)))

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        return ms(t0)

    for name in args.scenes:
        kw, spp, depth = SCENES[name]
        scene, camera, _ = T.scenes.tessellated(**kw, builder="sah")
        items = [p for _, p in scene.aggregate.items]
        flat = scene.flatten()
        nb = len(flat.tri_vertices)
        ids = np.zeros(nb, np.int32)
        ids[flat.prims["index"].astype(np.int64)] = flat.prims["material"]
        base_dev = [torch.from_numpy(np.ascontiguousarray(a)).cuda(0) for a in (flat.tri_vertices, flat.tri_normals, flat.tri_flags, ids)]
        film = cam = fd = None
        if name == "tess-1M":
            H, W = camera.film.pixels.shape[:2]
            film = torch.zeros((H, W, 4), dtype=torch.float32, device="cuda:0")
            cam, fd = camera.pod(), camera.film.desc()

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

        for mname, (stacks, slices) in MESHES.items():
            v, nrm, idx = T.scenes._uv_sphere(CENTER, RADIUS, stacks, slices)
            tri = idx.astype(np.int64).reshape(-1, 3) - 1
            mv, mn = torch.from_numpy(v[tri]).cuda(0), torch.from_numpy(nrm[tri]).cuda(0)
            mf = torch.full((len(tri),), 2, dtype=torch.uint8, device="cuda:0")
            mk = lambda: T.DeviceMeshScene([], mv, [mirror], None, mn, mf)
            row = {"scene": name, "base_triangles": nb, "mesh": mname, "mesh_triangles": len(tri)}
            ctx = T.Context(0, stream=stream.cuda_stream)
            ctx.upload(scene)
            row["first_attach_ms"] = timed(lambda: ctx.upload(T.CompositeScene(scene, mk())))
            row["attach_ms_all"] = [timed(lambda: ctx.upload(T.CompositeScene(scene, mk()))) for _ in range(args.runs)]
            row["attach_ms"] = statistics.median(row["attach_ms_all"])
            ph = [profiled(lambda: ctx.upload(T.CompositeScene(scene, mk())), "scene attach mesh device") for _ in range(3)]
            row["phases_ms"] = {k: statistics.median(p[k] for p in ph) for k in ph[0]}
            # the same geometry as one DeviceMeshScene
            allv = torch.cat([base_dev[0], mv])
            alln = torch.cat([base_dev[1], mn])
            allf = torch.cat([base_dev[2], mf])
            alli = torch.cat([base_dev[3], torch.full((len(tri),), len(flat.materials), dtype=torch.int32, device="cuda:0")])
            mats = flat.materials + [mirror]
            whole = lambda: T.DeviceMeshScene(scene.lights, allv, mats, alli, alln, allf)
            dctx = T.Context(0, stream=stream.cuda_stream)
            dctx.upload(whole())
            row["device_upload_ms_all"] = [timed(lambda: dctx.upload(whole())) for _ in range(args.runs)]
            row["device_upload_ms"] = statistics.median(row["device_upload_ms_all"])
            if film is not None and mname == "100k":
                cs = T.CompositeScene(scene, mk())
                ctx.upload(cs)
                dctx.upload(whole())
                row["frame_ms"] = {"composed_sah_base": frame_ms(ctx), "device_upload_lbvh": frame_ms(dctx)}
                row["spp"], row["max_depth"], row["resolution"], row["frames"] = spp, depth, list(kw["res"]), args.frames
            dctx.close()
            # the host path: one tree over everything, built and packed on the host
            hctx = T.Context(0, stream=stream.cuda_stream)
            tset = T.TriangleSet(ident, T.TriangleMesh(ident.object_to_world, len(tri), idx.reshape(-1), len(v), v, nrm))
            t0 = time.perf_counter()
            hs = T.Scene(scene.lights, T.BVHAccel(items + [T.PrimitiveBatch(tset, mirror)], 1, builder="lbvh"))
            t1 = time.perf_counter()
            hctx.upload(hs)
            torch.cuda.synchronize()
            row["host_path_s"] = {"bvhaccel_s": t1 - t0, "upload_s": time.perf_counter() - t1}
            row["host_path_s"]["total"] = row["host_path_s"]["bvhaccel_s"] + row["host_path_s"]["upload_s"]
            hctx.close()
            ctx.close()
            del hs, allv, alln, allf, alli
            torch.cuda.empty_cache()
            print(json.dumps({k: v for k, v in row.items() if not k.endswith("_all")}), flush=True)
            result["rows"].append(row)
        del scene, items, flat, base_dev, film
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["hardware"]))


if __name__ == "__main__":
    main()
