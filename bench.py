#!/usr/bin/env python
"""bench.py — benchmark of the ray-tracing hot path.  BASELINE.json's metric has two halves, "Mrays/sec (closest-hit +
shadow)" and "SPPM iterations/sec"; one invocation measures one workload as THE line and (for the default workload)
carries the SPPM workloads as complete sub-lines under "sppm".

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload NAME] [--dump-outputs DIR]

Whitted workloads (metric Mrays/s; a step = one full render):
  tess-1M   BASELINE.json configs[2] (C3): 1920x1080, 16 spp, depth 5, 999 840 triangles, Glass/Matte/Mirror  [default]
  tess-10M  configs[4] (C5): 4096x4096, 64 spp, depth 8, 10 002 224 triangles (meant for 8 GPUs)
  tess-small  a smoke-sized version
SPPM workloads (metric iterations/s; a step = one iteration):
  sppm-shadows-1024      configs[1] (C2): docs/code/spheres.jl at 1024x1024, depth 5
  sppm-caustic-glass-d5 / -d8   configs[0] (C1): docs/code/caustic_glass.jl as shipped (depth 5) and at the README's depth 8
  sppm-caustic-moving    configs[3] (C4): one frame of docs/code/caustic_moving.jl, 1.25 M photons, two lights

value = whole-job throughput with scene, queues and film resident in HBM (K steps between barriers, CUDA events, max
over ranks).  e2e = the same metric through the host-buffer C ABI call (trace_render_whitted / trace_render_sppm): the
film / image crosses PCIe inside the timed region.  N > 1: launched by torch.distributed.run, one rank per GPU, scene
replicated; tiles / image rows / photons are sharded and the exchange steps (film sum; visible-point all-gather and
(Phi, M) all-reduce) run inside libtrace_cuda.so on its own NCCL communicator - torch.distributed only carries the
communicator id, the barriers and the max-over-ranks of the timings.

--impl reference: the CPU restatement of the reference (oracle/, C++, std::thread over tiles / photons, all host cores)
on the same workload; the product's native library is not loaded in that process.

--dump-outputs DIR: after the timed steps, rank 0 writes what each timed path handed its caller after its last timed step
as DIR/<name>.npy (float32): film_<workload>.npy, the Whitted film (H, W, 4: X, Y, Z, filter weight), and
image_<workload>.npy, the SPPM image (H, W, 3).  Scenes and seeds depend on the arguments only, so two builds run with
the same arguments can be compared output for output.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (scene kwargs, spp, depth)
    "tess-1M": (dict(cells=600, stacks=266, slices=264, res=(1920, 1080), window=((-50.0, -28.125), (50.0, 28.125))), 16, 5),
    "tess-10M": (dict(cells=1900, stacks=835, slices=834, res=(4096, 4096), window=((-50.0, -50.0), (50.0, 50.0))), 64, 8),
    "tess-small": (dict(cells=64, stacks=34, slices=32, res=(480, 270), window=((-50.0, -28.125), (50.0, 28.125))), 4, 5),
}
SPPM_WORKLOADS = {
    # name: (builder name, kwargs, iterations of one render as the reference script ships it)
    "sppm-shadows-1024": ("shadows", dict(resolution=1024), 100),
    "sppm-caustic-glass-d5": ("caustic_glass", dict(resolution=256, max_depth=5), 100),
    "sppm-caustic-glass-d8": ("caustic_glass", dict(resolution=256, max_depth=8), 100),
    "sppm-caustic-moving": ("caustic_moving", dict(resolution=1024), 25),
    "sppm-shadows-small": ("shadows", dict(resolution=96), 8),
}
DUMP_BYTES = 64_000_000                     # --dump-outputs: all files together, .npy headers included
METRIC_WHITTED = "Mrays/sec (closest-hit + shadow)"
METRIC_SPPM = "SPPM iterations/sec"
L2_NOTE_WHITTED = "inputs larger than L2 (ray queues + BVH > 126 MB per step)"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def load_profile_table(name):
    """Static ncu-derived numbers committed under profiles/ (DRAM bytes per launch, issue / lane utilisation)."""
    p = os.path.join(ROOT, "profiles", name)
    try:
        return json.load(open(p))
    except Exception:
        return {}


def dump_outputs(outputs, path):
    """Write {name: (H, W, C) array} as path/<name>.npy in float32, DUMP_BYTES in all.  Smallest first, each array gets at
    most an equal share of what is left; one larger than its share is replaced by a seeded sample of its pixels (rows of
    the (H * W, C) view, in raster order), the same sample for the same shape."""
    os.makedirs(path, exist_ok=True)
    items = sorted(outputs.items(), key=lambda kv: kv[1].nbytes)
    left = DUMP_BYTES
    for k, (name, a) in enumerate(items):
        a = np.ascontiguousarray(a, dtype=np.float32)
        share = left // (len(items) - k) - 1024                  # (room for the .npy header)
        if a.nbytes > share:
            px = a.reshape(a.shape[0] * a.shape[1], -1)
            keep = np.random.default_rng(0).choice(len(px), share // px[0].nbytes, replace=False)
            a = px[np.sort(keep)]
        f = os.path.join(path, name + ".npy")
        np.save(f, a)
        left -= os.path.getsize(f)


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md's clocks line), sampled in-process through
    NVML every few ms - the timed region is short and `nvidia-smi -lms` needs longer than that to start.
    Falls back to one nvidia-smi query when NVML is not importable."""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self.running = False
        self.th = None
        self.nvml = None

    def _handle(self):
        import pynvml
        pynvml.nvmlInit()
        self.nvml = pynvml
        try:
            import torch
            uuid = str(torch.cuda.get_device_properties(self.gpu).uuid)
            return pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        except Exception:
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.gpu]) if vis and vis.split(",")[self.gpu].isdigit() else self.gpu
            return pynvml.nvmlDeviceGetHandleByIndex(idx)

    def _loop(self):
        n = self.nvml
        bits = {"hw_slowdown": getattr(n, "nvmlClocksEventReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(n, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while self.running:
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
                get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
                mask = int(get(self.h))
                for name, bit in bits.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        try:
            self.h = self._handle()
            self.max_mhz = float(self.nvml.nvmlDeviceGetMaxClockInfo(self.h, self.nvml.NVML_CLOCK_SM))
            self.running = True
            self.th = threading.Thread(target=self._loop, daemon=True)
            self.th.start()
        except Exception:
            self.nvml = None

    def stop(self):
        if self.th:
            self.running = False
            self.th.join(timeout=2)
        if not self.sm:                      # no NVML: one nvidia-smi sample right after the timed region
            try:
                out = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits", "-i",
                                      str(self.gpu)], capture_output=True, text=True, timeout=10).stdout.strip().split(",")
                return {"sm_mhz": float(out[0]), "sm_max_mhz": float(out[1]), "reasons": [], "samples": 1, "source": "nvidia-smi after the run"}
            except Exception:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.sm), "source": "nvml, 5 ms period, during the timed region"}


# ------------------------------------------------------------------ workloads (shared by both arms: identical `config`)
def build_scene(T, workload, builder="reference"):
    kw, spp, depth = WORKLOADS[workload]
    scene, camera, _ = T.scenes.tessellated(**kw, builder=builder)
    return scene, camera, spp, depth


def build_sppm_scene(T, workload, builder="reference"):
    name, kw, n_iter = SPPM_WORKLOADS[workload]
    kw = dict(kw)
    if name != "shadows":
        kw["builder"] = builder
    scene, camera, ikw = getattr(T.scenes, name)(**kw)
    photons = int(ikw.get("photons_per_iteration", -1))
    if photons <= 0:
        photons = int(camera.film.crop_bounds.area())
    return scene, camera, dict(r0=float(ikw["initial_search_radius"]), max_depth=int(ikw["max_depth"]), photons=photons,
                               iterations_per_render=n_iter)


def whitted_config(workload, scene):
    kw, spp, depth = WORKLOADS[workload]
    return {"workload": f"whitted-{workload}", "spp": spp, "max_depth": depth, "resolution": list(kw["res"]),
            "triangles": int(scene.aggregate.n_primitives),
            "l2_policy": "smoke-sized workload: L2-resident, not a benchmark" if workload == "tess-small" else L2_NOTE_WHITTED}


def sppm_config(workload, scene, camera, p):
    h, w = camera.film.pixels.shape[:2]
    return {"workload": workload, "resolution": [int(w), int(h)], "photons_per_iteration": p["photons"], "max_depth": p["max_depth"],
            "initial_search_radius": p["r0"], "primitives": int(scene.aggregate.n_primitives), "lights": len(scene.lights),
            "l2_policy": ("per-iteration working set (ray / photon queues, visible points, hash grid: > 400 MB) larger than L2" if w * h >= 1 << 20
                          else "small image: the per-iteration working set fits L2 (the reference's own configuration)")}


# ------------------------------------------------------------------ --impl reference (CPU; no product library)
def reference_setup():
    """Route the tree build through the checker so that the product's native library never enters this process."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    import trace_jl_b200 as T
    from trace_jl_b200 import scene as S
    S.BVH_BUILD_HOOK = lambda bounds, max_prims, builder: oracle_lib.bvh_build(bounds, max_prims)[:2]
    return T, oracle_lib


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    T, oracle_lib = reference_setup()
    cores = os.cpu_count() or 1
    budget = 150.0                                  # seconds for the whole --steps K --warmup W run
    n_steps = args.steps + args.warmup
    note = "restated reference (C++ oracle, std::thread, all host cores), not Trace.jl itself: no Julia in this image"
    if args.workload in SPPM_WORKLOADS:
        scene, camera, p = build_sppm_scene(T, args.workload)
        osc = oracle_lib.OracleScene(scene.flatten())
        cam, fd = camera.pod(), camera.film.desc()
        h, w = camera.film.pixels.shape[:2]
        rgb = np.zeros((h, w, 3), np.float32)
        # a step = one iteration.  Bounded sample: renders of the first iteration(s) of the 100-iteration render
        t0 = time.time(); osc.render_sppm(cam, fd, p["r0"], p["max_depth"], 1, p["photons"], 1, rgb, threads=cores); one = time.time() - t0
        per_step = max(1, min(4, int(budget / max(one, 1e-3) / max(1, n_steps))))
        times = []
        for i in range(n_steps):
            t0 = time.time(); osc.render_sppm(cam, fd, p["r0"], p["max_depth"], per_step, p["photons"], 1 + i, rgb, threads=cores); dt = time.time() - t0
            if i >= args.warmup:
                times.append(dt / per_step)
        value = 1.0 / (sum(times) / len(times))
        sample = f"renders of {per_step} iteration(s) (the first iterations of the 100-iteration render), all {p['photons']} photons and all pixels"
        out = {"impl": "reference", "metric": METRIC_SPPM, "value": value, "unit": "it/s", "n_gpus": args.gpus, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": 1e3 / value, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
               "dtype": "f32", "data": "synthetic", "config": sppm_config(args.workload, scene, camera, p),
               "cpu_baseline": {"value": value, "unit": "it/s", "cores": cores, "kind": "port", "sample": sample},
               "e2e": {"value": value, "unit": "it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "note": note}
        print(json.dumps(out))
        return
    scene, camera, spp, depth = build_scene(T, args.workload)
    osc = oracle_lib.OracleScene(scene.flatten())
    cam, fd = camera.pod(), camera.film.desc()
    film = np.zeros_like(camera.film.pixels)
    from trace_jl_b200.distributed import n_sample_tiles
    total_tiles = n_sample_tiles(camera.film)
    # full frame per step when the run fits the budget, else a strided subset of the 16x16 sample tiles (stated in `sample`)
    probe = min(total_tiles, max(cores * 8, 256))
    t0 = time.time(); osc.render_whitted(cam, fd, spp, depth, 1, film, max_tiles=probe, threads=cores); dt = time.time() - t0
    est_full = dt * total_tiles / probe
    tiles = total_tiles if est_full * n_steps <= budget else max(probe, int(total_tiles * budget / (est_full * n_steps)))
    times, rays = [], []
    for i in range(n_steps):
        film[:] = 0
        t0 = time.time(); cnt = osc.render_whitted(cam, fd, spp, depth, 1 + i, film, max_tiles=tiles if tiles < total_tiles else 0, threads=cores); dt = time.time() - t0
        if i >= args.warmup:
            times.append(dt); rays.append(int(cnt[0]) + int(cnt[1]))
    value = sum(rays) / sum(times) / 1e6
    sample = (f"the full frame ({total_tiles} 16x16 sample tiles) per step" if tiles >= total_tiles else
              f"{tiles} of {total_tiles} 16x16 sample tiles (strided over the image) per step") + f", {spp} spp, depth {depth}"
    print(json.dumps({
        "impl": "reference", "metric": METRIC_WHITTED, "value": value, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": whitted_config(args.workload, scene),
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "note": note}))


# ------------------------------------------------------------------ GPU arm
class Env:
    """Process-wide state of the GPU arm: ranks, stream, context, communicator."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        import trace_jl_b200 as T
        from trace_jl_b200 import distributed as D
        self.torch, self.dist, self.T, self.D, self.args = torch, dist, T, D, args
        self.t_start = time.perf_counter()
        self.outputs = {}                                   # --dump-outputs: name -> array after the last timed step
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
        torch.cuda.set_device(self.local)
        self.dev = f"cuda:{self.local}"
        if self.world > 1:
            import datetime
            # (a rank that dies must not leave the others waiting in a barrier for NCCL's default 10 minutes)
            dist.init_process_group("nccl", device_id=torch.device(self.dev), timeout=datetime.timedelta(seconds=240))
        # one non-default stream for everything: the library's launches (and its NCCL collectives) and the CUDA events
        # below share it (torch's default stream has handle 0, which the library takes as "make your own")
        self.stream = torch.cuda.Stream(device=self.local)
        torch.cuda.set_stream(self.stream)
        self.ctx = T.Context(self.local, stream=self.stream.cuda_stream)
        D.init_comm(self.ctx, self.rank, self.world)          # the library's own communicator (trace_comm_init)
        for k in ("slab", "walk", "lanes", "graph"):
            self.ctx.set_option(k, getattr(args, k))
        for kv in (args.option or []):                     # experiments: any trace_set_option key=value
            k, v = kv.split("=")
            self.ctx.set_option(k, int(v))
        if args.batch:
            self.ctx.set_option("batch", args.batch)

    def note(self, msg):
        """progress line on stderr (TRACE_BENCH_VERBOSE=1): which stage a rank reached, for post-mortems of multi-rank runs"""
        if os.environ.get("TRACE_BENCH_VERBOSE"):
            print(f"[bench rank {self.rank} +{time.perf_counter() - self.t_start:7.1f}s] {msg}", file=sys.stderr, flush=True)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([float(x)], device=self.dev, dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, xs):
        t = self.torch.tensor([float(x) for x in xs], device=self.dev, dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return [float(v) for v in t.tolist()]

    def timed(self, fn, steps):
        """EXACTLY `steps` calls of fn(i) between barriers, CUDA events on the shared stream; ms = max over ranks."""
        e0, e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
        self.barrier()
        t0 = time.perf_counter()
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        self.barrier()
        wall = (time.perf_counter() - t0) * 1e3
        return self.max_over_ranks(e0.elapsed_time(e1)), self.max_over_ranks(wall)


def kinds(st):
    from trace_jl_b200 import _lib
    return {n: (st["ms_kind"][i], st["launches_kind"][i]) for i, n in enumerate(_lib.KIND_NAMES)}


def bench_whitted(env, workload, with_extras=True):
    args, T, D, torch, ctx = env.args, env.T, env.D, env.torch, env.ctx
    world, rank = env.world, env.rank
    scene, camera, spp, depth = build_scene(T, workload, args.builder)
    flat = ctx.upload(scene)
    H, W = camera.film.pixels.shape[:2]
    film_dev = torch.zeros((H, W, 4), dtype=torch.float32, device=env.dev)
    film_bytes = film_dev.numel() * 4
    cam_pod, fd = camera.pod(), camera.film.desc()

    def step(i):                      # the film accumulates over the steps, as a reference film does over renders
        ctx.check(ctx.lib.trace_render_whitted_device(ctx.h, C.byref(cam_pod), C.byref(fd), spp, depth, C.c_uint64(1000 + i),
                                                      C.c_void_p(film_dev.data_ptr())))

    # ---- device-resident timing: W warm-up steps, then exactly K steps between barriers; max over ranks.  Multi-rank:
    # film_mode 0 = "tiles gathered once at the end": the library sums the ranks' films onto rank 0 (ncclReduce)
    ctx.set_option("film_mode", 0)
    ctx.set_option("time_kernels", 0)
    for i in range(args.warmup):
        step(i)
    env.barrier()
    ctx.reset_stats()
    sampler = ClockSampler(env.local)
    if rank == 0:
        sampler.start()
    ms_total, _ = env.timed(lambda i: step(args.warmup + i), args.steps)
    st = ctx.stats()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:              # (later passes keep accumulating into the same film)
        env.outputs[f"film_{workload}"] = film_dev.cpu().numpy()
    rays_e, rays_s, launches, prim_rays, prim_hits = env.sum_over_ranks(
        [st["rays_extend"], st["rays_shadow"], st["kernel_launches"], st["primary_rays"], st["primary_hits"]])
    total_rays = rays_e + rays_s
    value = total_rays / (ms_total * 1e-3) / 1e6
    hit_fraction = prim_hits / max(1.0, prim_rays)
    # rays that do real work: everything but the camera rays that leave the scene after a handful of box tests
    value_hit_only = (total_rays - (prim_rays - prim_hits)) / (ms_total * 1e-3) / 1e6

    # ---- roofline of the dominant kernel (closest-hit `extend`, incl. the fused primary stage): algorithmic bytes over the
    # CUDA-event launch time.  In the timed region up to `lanes` sub-batches run concurrently, so per-launch durations
    # are taken in a second timed pass with lanes = 1 (kernels back to back on one stream, events around every launch).
    ctx.set_option("lanes", 1)
    ctx.set_option("time_kernels", 1)
    step(5_000)
    env.barrier()
    ctx.reset_stats()
    serial_ms, _ = env.timed(lambda i: step(5_001 + i), args.steps)
    st1 = ctx.stats()
    kk = kinds(st1)
    ext_ms, ext_n = kk["extend"][0], max(1, kk["extend"][1])
    ctx.set_option("time_kernels", 0)
    ctx.set_option("count_nodes", 1)
    ctx.reset_stats()
    step(10_000)                                    # instrumented pass (not timed): box tests / primitive tests per ray
    torch.cuda.synchronize()
    sc = ctx.stats()
    ctx.set_option("count_nodes", 0)
    ctx.set_option("lanes", args.lanes)
    n_cnt = max(1, sc["rays_extend"] + sc["rays_shadow"])
    nodes_per_ray, prims_per_ray = sc["nodes_visited"] / n_cnt, sc["prims_tested"] / n_cnt
    bytes_per_ray = 48.0 + 32.0 * nodes_per_ray + 48.0 * prims_per_ray          # SURVEY.md §8d
    achieved = (st1["rays_extend"] * bytes_per_ray) / max(1e-9, ext_ms * 1e-3) / 1e9
    peak, peak_kind = load_peaks()
    prof = load_profile_table("extend_traffic.json")
    lim = prof.get("limits", {}).get(workload, {})
    roofline = {
        "bound": "issue",      # ncu: instruction issue at ~66 % of cycles with 22 of 32 lanes active - NOT HBM (dram_frac below)
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "rate": "algorithmic bytes (48 + 32 x box tests + 48 x primitive tests per ray) over the launch time, against the HBM copy peak; "
                "most of those bytes are L1 / L2 hits, see dram_frac",
        "traffic": prof.get(workload), "kernel": "k_wh_primary + k_wh_extend (pair-node walk)", "peak_source": f"of {peak_kind}",
        "avg_launch_ms": ext_ms / ext_n, "launches_timed": int(ext_n), "algorithmic_bytes_per_ray": bytes_per_ray,
        "box_tests_per_ray": nodes_per_ray, "prim_tests_per_ray": prims_per_ray,
        "extend_Mrays_per_s": st1["rays_extend"] / max(1e-9, ext_ms * 1e-3) / 1e6,
        "share_of_step": {k: v[0] / max(1e-9, serial_ms) for k, v in kk.items() if v[1]},
        "serial_pass_ms_per_step": serial_ms / args.steps,
        "issue_slots_busy_frac": lim.get("issue_active"), "lanes_active_of_32": lim.get("lanes"),
        "ncu_source": lim.get("source")}
    if roofline["traffic"]:
        roofline["dram_achieved_GBps"] = float(roofline["traffic"]) / (roofline["avg_launch_ms"] * 1e-3) / 1e9
        roofline["dram_frac"] = roofline["dram_achieved_GBps"] / peak

    # ---- per-rank breakdown (separate pass): render of the rank's tiles + the film sum, device time per rank
    breakdown = None
    if world > 1:
        parts = []
        for i in range(3):
            step(20_000 + i)
            torch.cuda.synchronize()
            parts.append(ctx.stats()["ms_total"])
        r = float(np.mean(parts))
        breakdown = {"render_plus_reduce_ms_max_over_ranks": env.max_over_ranks(r), "render_plus_reduce_ms_min_over_ranks": -env.max_over_ranks(-r)}

    # ---- e2e: the reference-facing C ABI call with HOST buffers (pinned), H2D + D2H inside the timed region.
    # Multi-rank: film_mode 1 - every rank uploads, merges and downloads its band of the film (N PCIe links instead of one)
    host_film = torch.zeros((H, W, 4), dtype=torch.float32).pin_memory()
    if world > 1:
        ctx.set_option("film_mode", 1)

    def e2e_step(i):
        ctx.check(ctx.lib.trace_render_whitted(ctx.h, C.byref(cam_pod), C.byref(fd), spp, depth, C.c_uint64(2000 + i),
                                               C.c_void_p(host_film.data_ptr())))

    for i in range(2):
        e2e_step(i)
    env.barrier()
    ctx.reset_stats()
    ms2, wall2 = env.timed(lambda i: e2e_step(2 + i), args.steps)
    st2 = ctx.stats()
    rays2 = sum(env.sum_over_ranks([st2["rays_extend"], st2["rays_shadow"]]))
    e2e_ms = max(ms2, wall2)
    cam_bytes = C.sizeof(cam_pod) + C.sizeof(fd)
    e2e = {"value": rays2 / (e2e_ms * 1e-3) / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": int(film_bytes + world * cam_bytes),
           "d2h_bytes_per_step": int(film_bytes), "ms_per_step": e2e_ms / args.steps,
           "film_delivery": "whole film on the one GPU" if world == 1 else
                            f"bands: rank r uploads, merges and downloads film pixels [r, r+1) x ceil(n / {world}) (option film_mode = 1)"}
    ctx.set_option("film_mode", 0)

    out = {"metric": METRIC_WHITTED, "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic", "config": whitted_config(workload, scene),
           "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
           "details": {"bvh_nodes": int(len(flat.nodes)),
                       "bvh_builder": {"reference": "reference split logic (src/accel/bvh.jl:87-185), bit-identical tree",
                                       "sah": "opt-in conventional binned SAH (same hits, ties aside)"}[args.builder],
                       "slab_test": {0: "literal (bounds.jl:180-200)", 1: "textbook (not hit-equivalent)",
                                     2: "guarded (literal AND conservative interval; hit-identical, tests/test_gpu_parity.py)"}[args.slab],
                       "walk": {1: "pair nodes (both children's boxes per fetch; bit-identical hits)", 0: "one node per step (bvh.jl:221-257)"}[args.walk],
                       "parallelism": f"tiles round-robin over {world} rank(s), film summed by the library (ncclReduce to rank 0)",
                       "lanes": args.lanes, "rays_per_step": total_rays / args.steps,
                       "primary_hit_fraction": hit_fraction, "Mrays_per_s_without_missing_camera_rays": value_hit_only},
           "breakdown": breakdown}

    # ---- the same workload on the OPT-IN tree (SURVEY.md 8f.2): same hits (t bit-identical, primitives equal except ties),
    # fewer box tests.  Reported next to the headline, which stays on the reference's own tree.
    if with_extras and args.builder == "reference" and not args.no_optin:
        scene2, camera2, _, _ = build_scene(T, workload, "sah")
        ctx.upload(scene2)
        for i in range(args.warmup):
            step(i)
        env.barrier()
        ctx.reset_stats()
        ms4, _ = env.timed(lambda i: step(args.warmup + i), args.steps)
        st4 = ctx.stats()
        rays4 = sum(env.sum_over_ranks([st4["rays_extend"], st4["rays_shadow"]]))
        out["optin_sah_tree"] = {"bvh_builder": "opt-in conventional binned SAH (trace_bvh_build_sah)", "value": rays4 / (ms4 * 1e-3) / 1e6,
                                 "unit": "Mrays/s", "ms_per_step": ms4 / args.steps, "bvh_nodes": int(len(scene2.flatten().nodes))}
        ctx.upload(scene)

    # ---- CPU baseline (rank 0, N = 1 only): the oracle on a bounded sample of the same workload
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib
        osc = oracle_lib.OracleScene(flat)
        cores = os.cpu_count() or 1
        tmp = np.zeros_like(camera.film.pixels)
        total_tiles = D.n_sample_tiles(camera.film)
        probe = min(total_tiles, max(cores * 8, 256))
        t0 = time.time(); osc.render_whitted(cam_pod, fd, spp, depth, 1, tmp, max_tiles=probe, threads=cores); dt = time.time() - t0
        tiles2 = int(min(total_tiles, max(probe, probe * 12.0 / max(dt, 1e-3))))
        t0 = time.time(); cnt = osc.render_whitted(cam_pod, fd, spp, depth, 1, tmp, max_tiles=tiles2 if tiles2 < total_tiles else 0, threads=cores); dt = time.time() - t0
        out["cpu_baseline"] = {"value": (int(cnt[0]) + int(cnt[1])) / dt / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port",
                               "sample": f"{tiles2} of {total_tiles} 16x16 sample tiles (strided over the image), {spp} spp, depth {depth}, {dt:.1f} s",
                               "note": "restated reference (C++ oracle, std::thread over tiles), not Trace.jl itself"}
    else:
        out["cpu_baseline"] = None
    return out


def bench_sppm(env, workload, steps, warmup, cpu_baseline=True):
    """One SPPM workload as a complete line: value (device-resident iterations), e2e (trace_render_sppm with a host image),
    roofline of its dominant kernel class, cpu_baseline (N = 1)."""
    args, T, D, torch, ctx = env.args, env.T, env.D, env.torch, env.ctx
    world, rank = env.world, env.rank
    scene, camera, p = build_sppm_scene(T, workload, args.builder)
    flat = ctx.upload(scene)
    h, w = camera.film.pixels.shape[:2]
    cam_pod, fd = camera.pod(), camera.film.desc()
    ctx.set_option("time_kernels", 0)
    env.note(f"{workload}: scene uploaded")
    sess = D.SPPMSession(ctx, scene, camera, p["r0"], p["max_depth"], p["photons"], 0x5EED0001)
    sess.step(max(3, warmup))
    env.barrier()
    env.note(f"{workload}: warm-up done")
    ctx.reset_stats()
    sampler = ClockSampler(env.local)
    if rank == 0:
        sampler.start()
    # the K timed iterations are handed to the library in ONE call (trace_sppm_iterate(first, K)): it enqueues them back to
    # back and, knowing what comes next, issues iteration it + 1's all-gather ahead of iteration it's all-reduce
    ms, _ = env.timed(lambda i: sess.step(steps), 1)
    clocks = sampler.stop() if rank == 0 else None
    st = ctx.stats()
    if args.dump_outputs:                           # (every rank: with several ranks the image is an all-gather)
        env.outputs[f"image_{workload}"] = sess.image()
    launches = sum(env.sum_over_ranks([st["kernel_launches"]]))
    value = steps / (ms * 1e-3)
    env.note(f"{workload}: timed iterations done ({value:.0f} it/s)")
    # serial pass with per-class CUDA events + counters: which kernel class dominates, and its algorithmic bytes
    ctx.set_option("time_kernels", 1)
    sess.step(1)
    ctx.synchronize()
    ctx.reset_stats()
    n_prof = min(steps, 8)
    ms_prof, _ = env.timed(lambda i: sess.step(n_prof), 1)
    img = sess.image()                      # (waits; also reports queue / grid overflows)
    s1 = ctx.stats()
    ctx.set_option("time_kernels", 0)
    sess.close()
    env.note(f"{workload}: per-class timing pass done")
    kk = kinds(s1)
    # the dominant class decides which extra passes (with collectives) follow: every rank must pick the SAME one, so the
    # choice is made on the class times summed over the ranks, not on this rank's own
    names = sorted(kk)
    summed = dict(zip(names, env.sum_over_ranks([kk[k][0] for k in names])))
    timed_total = sum(summed.values()) or 1e-9
    share = {k: summed[k] / timed_total for k in names if kk[k][1]}
    dom = max(share, key=share.get)
    peak, peak_kind = load_peaks()
    rays = s1["rays_extend"] + s1["rays_shadow"]
    if dom in ("extend", "shadow"):
        # traversal: same formula as the Whitted line; box / primitive tests per ray from an instrumented iteration
        ctx.set_option("count_nodes", 1)
        s2 = D.SPPMSession(ctx, scene, camera, p["r0"], p["max_depth"], p["photons"], 0x5EED0001)
        ctx.reset_stats()
        s2.step(1)
        ctx.synchronize()
        sc = ctx.stats()
        s2.close()
        ctx.set_option("count_nodes", 0)
        env.note(f"{workload}: counting pass done")
        n_cnt = max(1, sc["rays_extend"] + sc["rays_shadow"])
        npr, ppr = sc["nodes_visited"] / n_cnt, sc["prims_tested"] / n_cnt
        per_unit = 48.0 + 32.0 * npr + 48.0 * ppr
        units = s1["rays_extend"] if dom == "extend" else s1["rays_shadow"]
        detail = {"kernel": "k_wh_extend (closest hit, camera + photon paths)" if dom == "extend" else "k_wh_shadow",
                  "algorithmic_bytes_per_ray": per_unit, "box_tests_per_ray": npr, "prim_tests_per_ray": ppr}
    elif dom == "deposit":
        # SURVEY.md §8d: per deposit request 48 B (p, wo, beta) + 8 B cell range + 16 B per candidate + per accepted
        # visible point 4 B index + 64 B record + 16 B atomic
        req, cand, dep = s1["sppm_requests"], s1["sppm_candidates"], s1["sppm_deposits"]
        units = max(1, req)
        per_unit = (56.0 * req + 16.0 * cand + 84.0 * dep) / units
        detail = {"kernel": "k_photon_deposit", "algorithmic_bytes_per_request": per_unit, "candidates_per_request": cand / units,
                  "deposits_per_request": dep / units}
    elif dom == "grid":
        # per iteration: 3 passes over the visible points (bounds, count, fill: 32 B each) + per (visible point, cell)
        # entry 4 B count atomic + 4 B cursor atomic + 20 B written, + 3 passes over the cell table (scan)
        items = s1["sppm_grid_items"]
        units = max(1, items)
        n_it = max(1, kk["grid"][1])
        per_unit = (28.0 * items + n_it * (96.0 * w * h + 24.0 * w * h)) / units
        detail = {"kernel": "k_grid_bounds / k_grid_insert<count, fill> / scan", "algorithmic_bytes_per_grid_entry": per_unit,
                  "grid_entries_per_iteration": items / n_it}
    else:
        # shade / generate / update: streaming kernels over the ray queues
        units = max(1, rays)
        per_unit = {"shade": 16.0 + 48.0 + 48.0 + 96.0 + 48.0, "generate": 48.0, "update": 56.0}.get(dom, 64.0)
        detail = {"kernel": dom, "algorithmic_bytes_per_ray": per_unit}
    achieved = units * per_unit / max(1e-9, kk[dom][0] * 1e-3) / 1e9
    prof = load_profile_table("sppm_traffic.json").get(workload, {})
    roofline = {"bound": "hbm" if dom in ("deposit", "grid", "shade", "generate", "update") else "issue",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": prof.get(dom),
                "peak_source": f"of {peak_kind}", "dominant_class": dom, "avg_launch_ms": kk[dom][0] / max(1, kk[dom][1]),
                "launches_timed": int(kk[dom][1]), "share_of_kernel_time": share,
                "serial_ms_per_iteration": ms_prof / n_prof, **detail}
    if roofline["traffic"]:
        roofline["dram_achieved_GBps"] = float(roofline["traffic"]) / (roofline["avg_launch_ms"] * 1e-3) / 1e9
        roofline["dram_frac"] = roofline["dram_achieved_GBps"] / peak

    # ---- e2e: trace_render_sppm, the call the Julia functor makes: n iterations + the image into a HOST buffer
    # (iterations per render: the scene script's own count up to 25 - caustic_moving renders exactly its 25-iteration frame)
    n_it = int(min(p["iterations_per_render"], 25))
    rgb = torch.zeros((h, w, 3), dtype=torch.float32).pin_memory()

    def render(i):
        ctx.check(ctx.lib.trace_render_sppm(ctx.h, C.byref(cam_pod), C.byref(fd), p["r0"], p["max_depth"], n_it, p["photons"], 0,
                                            C.c_uint64(0x5EED0001 + i), C.cast(None, T._lib.SPPM_CB), None, C.c_void_p(rgb.data_ptr())))

    render(0)
    env.note(f"{workload}: first e2e render done")
    n_renders = 3
    ms_e, wall_e = env.timed(lambda i: render(1 + i), n_renders)
    e2e_ms = max(ms_e, wall_e)
    env.note(f"{workload}: e2e renders done")
    e2e = {"value": n_renders * n_it / (e2e_ms * 1e-3), "unit": "it/s",
           "h2d_bytes_per_step": int(world * (C.sizeof(cam_pod) + C.sizeof(fd)) / n_it), "d2h_bytes_per_step": int(world * h * w * 3 * 4 / n_it),
           "ms_per_step": e2e_ms / (n_renders * n_it),
           "what": f"trace_render_sppm: renders of {n_it} iterations each (session set-up, {n_it} iterations, image to a pinned host buffer on every rank)"}
    out = {"metric": METRIC_SPPM, "value": value, "unit": "it/s", "n_gpus": world, "steps": steps, "warmup": max(3, warmup),
           "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic", "config": sppm_config(workload, scene, camera, p), "e2e": e2e, "gpu_launches": int(launches),
           "clocks": clocks, "roofline": roofline,
           "details": {"image_mean": float(img.mean()), "parallelism": (f"camera paths by image rows, photons by index range over {world} ranks; "
                       "visible-point all-gather + (Phi, M) all-reduce per iteration inside the library") if world > 1 else "one GPU"}}
    if rank == 0 and world == 1 and cpu_baseline and not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib
        osc = oracle_lib.OracleScene(flat)
        cores = os.cpu_count() or 1
        ref = np.zeros((h, w, 3), np.float32)
        t0 = time.time(); osc.render_sppm(cam_pod, fd, p["r0"], p["max_depth"], 1, p["photons"], 1, ref, threads=cores); one = time.time() - t0
        n_cpu = int(max(1, min(6, 8.0 / max(one, 1e-3))))
        t0 = time.time(); osc.render_sppm(cam_pod, fd, p["r0"], p["max_depth"], n_cpu, p["photons"], 1, ref, threads=cores); dt = time.time() - t0
        out["cpu_baseline"] = {"value": n_cpu / dt, "unit": "it/s", "cores": cores, "kind": "port",
                               "sample": f"the first {n_cpu} iteration(s) of the render, all photons and pixels, {dt:.1f} s",
                               "note": "restated reference (C++ oracle, std::thread), not Trace.jl itself"}
    else:
        out["cpu_baseline"] = None
    return out


def sppm_sharding_check(env):
    """N > 1 self-check on the real collectives: a small render over all ranks against the same render on rank 0 alone
    (second context, no communicator); the sharding must not change the image beyond the order of the float flux atomics."""
    T, ctx = env.T, env.ctx
    scene, camera, kw = T.scenes.shadows(resolution=160)
    h, w = camera.film.pixels.shape[:2]
    cam, fd = camera.pod(), camera.film.desc()
    ctx.upload(scene)
    a = np.zeros((h, w, 3), np.float32)
    ctx.check(ctx.lib.trace_render_sppm(ctx.h, C.byref(cam), C.byref(fd), kw["initial_search_radius"], kw["max_depth"], 4, -1, 0,
                                        C.c_uint64(0x5EED0001), C.cast(None, T._lib.SPPM_CB), None, T._lib.ptr(a)))
    check = None
    if env.rank == 0:
        solo = T.Context(env.local, stream=env.stream.cuda_stream)
        solo.upload(scene)
        b = np.zeros_like(a)
        solo.check(solo.lib.trace_render_sppm(solo.h, C.byref(cam), C.byref(fd), kw["initial_search_radius"], kw["max_depth"], 4, -1, 0,
                                              C.c_uint64(0x5EED0001), C.cast(None, T._lib.SPPM_CB), None, T._lib.ptr(b)))
        solo.close()
        check = {"workload": "sppm-shadows-160, 4 iterations, trace_render_sppm over all ranks vs one GPU",
                 "max_abs_diff_vs_one_gpu": float(np.abs(a - b).max()), "image_max": float(b.max()),
                 "ok": bool(np.allclose(a, b, rtol=3e-4, atol=1e-6))}
    env.barrier()
    return check


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--workload", default="tess-1M", choices=sorted(WORKLOADS) + sorted(SPPM_WORKLOADS))
    ap.add_argument("--slab", type=int, default=2)
    ap.add_argument("--walk", type=int, default=1, help="traversal loop: 1 pair nodes (default), 0 one node per step (the reference loop)")
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--lanes", type=int, default=12)
    ap.add_argument("--builder", default="reference", choices=["reference", "sah"],
                    help="BVH build: the reference's split logic (default, bit-identical tree) or the opt-in conventional SAH")
    ap.add_argument("--graph", type=int, default=1, help="replay the Whitted render as one CUDA graph (0: direct launches)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sppm", action="store_true")
    ap.add_argument("--option", action="append", help="extra trace_set_option key=value (experiments), repeatable")
    ap.add_argument("--no-optin", action="store_true", help="skip the extra measurement on the opt-in SAH tree")
    ap.add_argument("--sppm-workloads", default="sppm-shadows-1024,sppm-caustic-moving,sppm-caustic-glass-d8",
                    help="SPPM sub-lines carried by the default Whitted line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32, 64 MB in all; GPU arm)")
    args = ap.parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of the GPU arm; it has no meaning with --impl reference")
        return run_reference(args)
    env = Env(args)
    if args.workload in SPPM_WORKLOADS:
        out = bench_sppm(env, args.workload, args.steps, args.warmup)
        if env.world > 1:
            out["sharded_vs_single_gpu_check"] = sppm_sharding_check(env)
    else:
        out = bench_whitted(env, args.workload)
        if not args.no_sppm:
            # the metric's second half: every SPPM workload as a complete line of its own (value, e2e, roofline, cpu_baseline),
            # K timed iterations each (with sppm_pipeline iterations in flight, fill and drain are part of the timed region)
            out["sppm"] = [bench_sppm(env, wl, args.steps, args.warmup, cpu_baseline=True) for wl in args.sppm_workloads.split(",") if wl]
            if env.world > 1:
                out["sppm"].append({"sharded_vs_single_gpu_check": sppm_sharding_check(env)})
    if env.rank == 0:
        if args.dump_outputs:
            dump_outputs(env.outputs, args.dump_outputs)
        print(json.dumps(out))
    env.ctx.close()
    if env.world > 1:
        env.dist.destroy_process_group()


if __name__ == "__main__":
    main()
