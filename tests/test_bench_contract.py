"""bench.py contract pieces that can be checked without a GPU: the reference arm prints one JSON line with the agreed keys
(it times the CPU restatement on a bounded sample), ranks other than 0 stay silent, and our own arm refuses to run
without a CUDA device instead of falling back to anything.  With a GPU (-m gpu): --dump-outputs writes what the timed
steps computed."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, env=e, capture_output=True, text=True,
                          timeout=600)


def test_reference_arm_prints_the_contract_line():
    r = _run(["--impl", "reference", "--workload", "tess-small", "--steps", "2", "--warmup", "1"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Mrays/s" and d["higher_is_better"] is True
    assert d["metric"] == "Mrays/sec (closest-hit + shadow)" and d["steps"] == 2 and d["warmup"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "tiles" in d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"] == "whitted-tess-small"


def test_reference_arm_other_ranks_are_silent():
    r = _run(["--impl", "reference", "--workload", "tess-small", "--steps", "1", "--warmup", "1"], env={"RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_our_arm_needs_a_gpu():
    r = _run(["--workload", "tess-small", "--steps", "1", "--warmup", "3"])
    assert r.returncode != 0
    assert "no CPU fallback" in (r.stderr + r.stdout)


def test_reference_arm_covers_the_sppm_half_of_the_metric():
    r = _run(["--impl", "reference", "--workload", "sppm-shadows-small", "--steps", "2", "--warmup", "1"])
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert d["impl"] == "reference" and d["metric"] == "SPPM iterations/sec" and d["unit"] == "it/s" and d["value"] > 0
    assert d["config"]["workload"] == "sppm-shadows-small" and d["config"]["photons_per_iteration"] == 95 * 95
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["cpu_baseline"]["kind"] == "port"


def test_reference_arm_never_loads_the_product_library():
    """--impl reference must time the checker alone: scene description in Python, tree build and render in oracle/ -
    libtrace_cuda.so must not be mapped into that process (VERDICT r1: native_so_loaded listed it)."""
    code = (
        "import sys; sys.path.insert(0, %r); import bench\n"
        "T, o = bench.reference_setup()\n"
        "scene, camera, spp, depth = bench.build_scene(T, 'tess-small')\n"
        "osc = o.OracleScene(scene.flatten())\n"
        "s2, c2, p = bench.build_sppm_scene(T, 'sppm-caustic-glass-d5')\n"
        "s2.flatten()\n"
        "maps = open('/proc/self/maps').read()\n"
        "assert 'libtrace_ref' in maps and 'libtrace_cuda' not in maps, [l for l in maps.splitlines() if 'libtrace' in l]\n"
        "print('clean')\n") % ROOT
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "clean" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_both_arms_share_one_config():
    """The driver compares the arms' `config`: both must come from the same function of the workload alone."""
    sys.path.insert(0, ROOT)
    import bench
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert src.count('"config": whitted_config(') == 2 and src.count('"config": sppm_config(') == 2


def test_dump_outputs_budget_and_sample(tmp_path):
    """Outputs that fit are written whole; one that does not is replaced by the same seeded sample of whole pixels on
    every run, and all files together stay within DUMP_BYTES."""
    sys.path.insert(0, ROOT)
    import bench
    big = np.random.default_rng(3).random((2048, 2048, 4), dtype=np.float32)      # 64 MiB on its own
    big[..., 0] = np.arange(2048 * 2048, dtype=np.float32).reshape(2048, 2048)     # channel 0 names the pixel
    small = np.random.default_rng(4).random((64, 48, 3), dtype=np.float32)
    for d in ("a", "b"):
        bench.dump_outputs({"big": big, "small": small}, str(tmp_path / d))
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["big.npy", "small.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_BYTES
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), small)
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert a.dtype == np.float32 and a.shape[1] == 4 and len(a) > 3_000_000 and np.array_equal(a, b)
    idx = a[:, 0].astype(np.int64)
    assert np.all(np.diff(idx) > 0) and np.array_equal(a, big.reshape(-1, 4)[idx])


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(T, tmp_path):
    """The dumped Whitted film is the film after warm-up + K renders (seeds 1000, 1001, ...; it accumulates), the dumped
    SPPM image the image after max(3, W) + K iterations; both equal the same work done directly through the library, up to
    the order of the float atomics."""
    steps, warmup = 3, 2
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tess-small", "--steps", str(steps),
                        "--warmup", str(warmup), "--no-cpu-baseline", "--no-optin", "--sppm-workloads", "sppm-shadows-small",
                        "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert d["steps"] == steps and d["sppm"][0]["steps"] == steps
    assert sorted(os.listdir(tmp_path)) == ["film_tess-small.npy", "image_sppm-shadows-small.npy"]
    sys.path.insert(0, ROOT)
    import bench
    from trace_jl_b200 import distributed as D
    ctx = T.Context(0)
    try:
        scene, camera, spp, depth = bench.build_scene(T, "tess-small")
        ctx.upload(scene)
        cam, fd = camera.pod(), camera.film.desc()
        want = np.zeros_like(camera.film.pixels)
        for i in range(warmup + steps):
            ctx.check(ctx.lib.trace_render_whitted(ctx.h, C.byref(cam), C.byref(fd), spp, depth, C.c_uint64(1000 + i), T._lib.ptr(want)))
        film = np.load(tmp_path / "film_tess-small.npy")
        assert film.dtype == np.float32 and film.shape == want.shape and float(want[..., 3].min()) > 0
        assert np.allclose(film, want, rtol=1e-5, atol=1e-6), float(np.abs(film - want).max())
        scene, camera, p = bench.build_sppm_scene(T, "sppm-shadows-small")
        sess = D.SPPMSession(ctx, scene, camera, p["r0"], p["max_depth"], p["photons"], 0x5EED0001)
        sess.step(max(3, warmup) + steps)
        want = sess.image()
        sess.close()
        img = np.load(tmp_path / "image_sppm-shadows-small.npy")
        assert img.dtype == np.float32 and img.shape == want.shape and float(want.max()) > 0
        assert np.allclose(img, want, rtol=2e-4, atol=1e-6), float(np.abs(img - want).max())
    finally:
        ctx.close()
