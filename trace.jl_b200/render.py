"""Host-side mirror of Trace.jl's sensing + integrator API: LanczosSincFilter (src/filter.jl), Film (src/film.jl),
PerspectiveCamera (src/camera/perspective.jl), UniformSampler (src/sampler/sampler.jl:129-151), WhittedIntegrator
(src/integrators/sampler.jl) and SPPMIntegrator (src/integrators/sppm.jl).  The integrators are functors on a Scene,
like the reference's; the render itself runs in libtrace_cuda.so through the C ABI (include/trace_cuda.h).
"""
import ctypes as C
import struct
import zlib

import numpy as np

from . import _lib
from .geometry import Bounds2, Point2f, Transformation, _v3, f32, perspective, scale, translate
from .scene import DeviceMeshScene


class LanczosSincFilter:
    """src/filter.jl:3-23"""

    def __init__(self, radius, tau):
        self.radius = Point2f(radius)
        self.tau = f32(tau)

    @staticmethod
    def _sinc(x):
        x = f32(abs(x))
        if x < f32(1e-5):
            return f32(1)
        x = f32(x * f32(np.pi))
        return f32(f32(np.sin(x)) / x)

    def _windowed(self, x, r):
        x = f32(abs(x))
        if x > r:
            return f32(0)
        return f32(self._sinc(x) * self._sinc(f32(x / self.tau)))

    def __call__(self, p):
        p = Point2f(p)
        return f32(self._windowed(p[0], self.radius[0]) * self._windowed(p[1], self.radius[1]))


class Film:
    """src/film.jl:7-62.  `pixels` is [crop_h, crop_w, 4] float32 = (X, Y, Z, filter_weight_sum) per pixel, indexed
    [y - crop_y0, x - crop_x0] (the reference's `pixels[y, x]`)."""

    def __init__(self, resolution, crop_bounds, filter, diagonal, scale, filename=None):
        self.resolution = Point2f(resolution)
        lo = np.ceil(self.resolution * crop_bounds.p_min) + f32(1)
        hi = np.ceil(self.resolution * crop_bounds.p_max)
        self.crop_bounds = Bounds2(lo, hi)
        sides = [int(s) for s in self.crop_bounds.inclusive_sides()]
        self.pixels = np.zeros((sides[1], sides[0], 4), dtype=np.float32)
        self.filter = filter
        self.diagonal = f32(f32(diagonal) * f32(0.001))
        self.filename = filename
        self.scale = f32(scale)
        self.filter_table_width = 16
        r = filter.radius / f32(16)
        tbl = np.zeros((16, 16), dtype=np.float32)
        for y in range(16):
            for x in range(16):
                tbl[y, x] = filter(Point2f(f32(f32(x + 0.5) * r[0]), f32(f32(y + 0.5) * r[1])))
        self.filter_table = tbl

    def get_sample_bounds(self):                     # :68-73
        return Bounds2(np.floor(self.crop_bounds.p_min + f32(0.5) - self.filter.radius),
                       np.ceil(self.crop_bounds.p_max - f32(0.5) + self.filter.radius))

    def desc(self):
        d = _lib.FilmDesc()
        d.crop_x0, d.crop_y0 = int(self.crop_bounds.p_min[0]), int(self.crop_bounds.p_min[1])
        d.crop_x1, d.crop_y1 = int(self.crop_bounds.p_max[0]), int(self.crop_bounds.p_max[1])
        d.filter_radius[0], d.filter_radius[1] = float(self.filter.radius[0]), float(self.filter.radius[1])
        C.memmove(d.filter_table, np.ascontiguousarray(self.filter_table, dtype=np.float32).ctypes.data, 256 * 4)
        d.scale = float(self.scale)
        return d

    def set_image(self, rgb):                        # set_image!, :195-202
        rgb = np.asarray(rgb, dtype=np.float32).reshape(self.pixels.shape[0], self.pixels.shape[1], 3)
        m = np.array([[0.412453, 0.357580, 0.180423], [0.212671, 0.715160, 0.072169], [0.019334, 0.119193, 0.950227]],
                     dtype=np.float32)
        self.pixels[..., :3] = rgb @ m.T
        self.pixels[..., 3] = 1.0

    def to_rgb(self):
        """The image `save` writes (film.jl:204-221): XYZ->RGB, / weight sum, max 0, * scale, clamp [0,1]; rows NOT
        yet flipped."""
        m = np.array([[3.240479, -1.537150, -0.498535], [-0.969256, 1.875991, 0.041556], [0.055648, -0.204043, 1.057311]],
                     dtype=np.float32)
        img = self.pixels[..., :3] @ m.T
        w = self.pixels[..., 3]
        nz = w != 0
        img[nz] = np.maximum(0.0, img[nz] * (f32(1) / w[nz])[:, None])
        img = img * self.scale
        return np.clip(img, 0.0, 1.0).astype(np.float32)

    def save(self, filename=None):
        filename = filename or self.filename
        img = self.to_rgb()[::-1]                    # rows flipped, film.jl:221
        if filename:
            write_png(filename, img)
        return img


def write_png(path, img01):
    """Minimal 8-bit RGB PNG encoder (PNG encode stays on the host, SURVEY.md §2)."""
    a = (np.clip(img01, 0, 1) * 255.0 + 0.5).astype(np.uint8)
    h, w, _ = a.shape
    raw = b"".join(b"\x00" + a[y].tobytes() for y in range(h))

    def chunk(tag, data):
        c = struct.pack(">I", len(data)) + tag + data
        return c + struct.pack(">I", zlib.crc32(tag + data) & 0xFFFFFFFF)

    with open(path, "wb") as fh:
        fh.write(b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, 2, 0, 0, 0)) +
                 chunk(b"IDAT", zlib.compress(raw, 6)) + chunk(b"IEND", b""))


class PerspectiveCamera:
    """src/camera/perspective.jl:1-81 (ProjectiveCamera + PerspectiveCamera)."""

    def __init__(self, camera_to_world, screen_window, shutter_open, shutter_close, lens_radius, focal_distance, fov, film):
        self.camera_to_world = camera_to_world
        self.shutter_open, self.shutter_close = f32(shutter_open), f32(shutter_close)
        self.lens_radius, self.focal_distance = f32(lens_radius), f32(focal_distance)
        self.film = film
        self.camera_to_screen = perspective(f32(fov), f32(0.01), f32(1000))
        sw = screen_window
        self.screen_to_raster = (
            scale(film.resolution[0], film.resolution[1], 1)
            * scale(f32(1) / f32(sw.p_max[0] - sw.p_min[0]), f32(1) / f32(sw.p_max[1] - sw.p_min[1]), 1)
            * translate(_v3([-sw.p_min[0], -sw.p_max[1], 0])))
        self.raster_to_screen = self.screen_to_raster.inv()
        self.raster_to_camera = self.camera_to_screen.inv() * self.raster_to_screen

    def get_film(self):
        return self.film

    def pod(self):
        c = _lib.Camera()
        r2c = self.raster_to_camera.m.reshape(-1)
        c2w = self.camera_to_world.m.reshape(-1)
        for i in range(16):
            c.raster_to_camera[i] = float(r2c[i])
            c.camera_to_world[i] = float(c2w[i])
        c.lens_radius, c.focal_distance = float(self.lens_radius), float(self.focal_distance)
        c.shutter_open, c.shutter_close = float(self.shutter_open), float(self.shutter_close)
        return c


class UniformSampler:
    """src/sampler/sampler.jl:129-133"""

    def __init__(self, samples_per_pixel):
        self.samples_per_pixel = int(samples_per_pixel)


# ------------------------------------------------------------------ device context
class Context:
    """One trace_ctx (one GPU).  `stream` may be a raw cudaStream_t of a NON-default stream (e.g. a torch.cuda.Stream's
    .cuda_stream); with None / 0 (torch's default stream has handle 0) the library creates its own non-blocking stream,
    which does not order against torch's work - `distributed.py` then fences with host synchronisation."""

    def __init__(self, device=0, stream=None):
        self.lib = _lib.load()
        self.device = int(device)
        self.h = C.c_void_p()
        self.stream_handle = int(stream) if stream else 0
        rc = self.lib.trace_create(C.byref(self.h), int(device), C.c_void_p(stream) if stream else None)
        if rc != 0:
            raise RuntimeError(f"trace_create failed ({rc}): no usable CUDA device; there is no CPU fallback")
        self._scene = None
        self._n_nodes = 0

    def check(self, rc):
        if rc != 0:
            msg = self.lib.trace_last_error(self.h)
            raise RuntimeError(f"libtrace_cuda error {rc}: {msg.decode() if msg else '?'}")

    def set_option(self, key, value):
        self.check(self.lib.trace_set_option(self.h, key.encode(), int(value)))

    # multi-GPU: the library's own NCCL communicator (include/trace_cuda.h, trace_comm_*)
    def comm_init(self, comm_id, rank, world):
        """Collective: every rank calls it with the SAME id (bytes from `comm_unique_id()` on rank 0)."""
        if len(comm_id) != _lib.COMM_ID_BYTES:
            raise ValueError("communicator id must be %d bytes" % _lib.COMM_ID_BYTES)
        buf = C.create_string_buffer(bytes(comm_id), _lib.COMM_ID_BYTES)
        self.check(self.lib.trace_comm_init(self.h, buf, int(rank), int(world)))

    def comm_destroy(self):
        self.check(self.lib.trace_comm_destroy(self.h))

    def comm_info(self):
        r, w, v = C.c_int(), C.c_int(), C.c_int()
        self.check(self.lib.trace_comm_info(self.h, C.byref(r), C.byref(w), C.byref(v)))
        return {"rank": r.value, "world": w.value, "nccl_version": v.value}

    def upload(self, scene):
        if isinstance(scene, DeviceMeshScene):
            if self._scene is not scene:
                self._upload_mesh(scene)
            return scene
        flat = scene.flatten()
        if self._scene is not flat:
            if flat.stale:
                raise RuntimeError("this scene was refit on a context and its host nodes / vertices are stale: upload it "
                                   "before refitting and refit every context with the same vertices, or build a new "
                                   "BVHAccel for the moved geometry")
            d = flat.desc()
            self.check(self.lib.trace_scene_upload(self.h, C.byref(d)))
            self._scene, self._n_nodes = flat, len(flat.nodes)
        return flat

    def _upload_mesh(self, scene):
        """trace_scene_upload_mesh_device: tree and scene buffers built on the GPU from the scene's device arrays"""
        d, keep = scene.desc(self.device)
        import torch
        torch.cuda.current_stream(self.device).synchronize()       # the work that wrote the arrays is done
        n_nodes = C.c_int64()
        self.check(self.lib.trace_scene_upload_mesh_device(self.h, C.byref(d), C.byref(n_nodes)))
        self._scene, self._n_nodes = scene, n_nodes.value

    def refit(self, scene, vertices=None, normals=None):
        """Move the triangles of the scene uploaded to this context and refit its tree on the GPU (trace_scene_refit):
        same topology, every box recomputed.  `vertices` is [n_tris, 3, 3] in the triangle order of the scene's
        flattening (`FlatScene.tri_vertices`):
          None                   the meshes' current `vertices` (move a mesh's vertices, then refit);
          numpy array            through host memory;
          float32 CUDA tensor    (contiguous, on this context's device) read in place on the GPU: no host traffic.
        `normals` (same layout and kind as `vertices`, or None to keep the current ones) apply to triangles uploaded
        with normals.  Afterwards the host FlatScene's nodes are stale: it cannot be uploaded to another context.
        A DeviceMeshScene: `vertices` in its triangle order; None re-reads the scene's own tensors (vertices, and
        normals if it has them) after the caller changed them in place."""
        if isinstance(scene, DeviceMeshScene):
            if scene is not self._scene:
                raise ValueError("refit: this scene is not the one uploaded to this context")
            flat, n, sb = None, scene.n_tris, np.zeros((0, 6), np.float32)
            if vertices is None:
                vertices = scene.vertices
            if normals is None and hasattr(vertices, "is_cuda"):
                normals = scene.normals
        else:
            flat = scene.flatten() if scene._flat is not None else None
            if flat is None or flat is not self._scene:
                raise ValueError("refit: this scene is not the one uploaded to this context")
            n = len(flat.tri_vertices)
            sb = np.ascontiguousarray(flat.sphere_bounds, dtype=np.float32)
            if vertices is None:
                vertices = flat.gather_vertices()
        sb_ptr = _lib.ptr(sb) if len(sb) else None
        if hasattr(vertices, "is_cuda"):                      # a torch tensor
            def dev_ptr(t, what):
                if t is None:
                    return None
                if not (hasattr(t, "is_cuda") and t.is_cuda and t.device.index == self.device):
                    raise ValueError(f"refit: {what} must be a CUDA tensor on device {self.device}")
                if str(t.dtype) != "torch.float32" or not t.is_contiguous() or t.numel() != 9 * n:
                    raise ValueError(f"refit: {what} must be a contiguous float32 tensor of {n} x 3 x 3")
                return t.data_ptr()
            vp, np_ = dev_ptr(vertices, "vertices"), dev_ptr(normals, "normals")
            import torch
            torch.cuda.current_stream(self.device).synchronize()    # the work that wrote them is done
            self.check(self.lib.trace_scene_refit_device(self.h, n, vp, np_, len(sb), sb_ptr))
        else:
            def host(a, what):
                if a is None:
                    return None
                a = np.ascontiguousarray(a, dtype=np.float32)
                if a.size != 9 * n:
                    raise ValueError(f"refit: {what} must be {n} x 3 x 3")
                return a
            v, nn = host(vertices, "vertices"), host(normals, "normals")
            self.check(self.lib.trace_scene_refit(self.h, n, _lib.ptr(v), _lib.ptr(nn), len(sb), sb_ptr))
        if flat is not None:
            flat.stale = True

    def scene_nodes(self):
        """The uploaded scene's nodes as the device holds them now (trace_scene_copy_nodes), node_dtype."""
        if self._scene is None:
            raise ValueError("no scene uploaded")
        nodes = np.zeros(self._n_nodes, dtype=_lib.node_dtype)
        self.check(self.lib.trace_scene_copy_nodes(self.h, _lib.ptr(nodes)))
        return nodes

    def shadow_tree(self):
        """The uploaded scene's shadow tree as its pair records (trace_scene_shadow_tree): float32 [n_prims - 1, 16]
        (viewed as uint32, columns 6, 7, 14, 15 are references and split-axis bits), or None when the scene has none."""
        n = C.c_int64()
        self.check(self.lib.trace_scene_shadow_tree(self.h, C.byref(n), None))
        if n.value == 0:
            return None
        pairs = np.zeros((n.value, 16), dtype=np.float32)
        self.check(self.lib.trace_scene_shadow_tree(self.h, C.byref(n), _lib.ptr(pairs)))
        return pairs

    def stats(self):
        s = _lib.Stats()
        self.check(self.lib.trace_get_stats(self.h, C.byref(s)))
        out = s.as_dict()
        fb = C.c_uint64()
        self.check(self.lib.trace_get_shadow_fallbacks(self.h, C.byref(fb)))
        out["shadow_fallbacks"] = fb.value
        return out

    def reset_stats(self):
        self.check(self.lib.trace_reset_stats(self.h))

    def synchronize(self):
        self.check(self.lib.trace_synchronize(self.h))

    def close(self):
        if self.h:
            self.lib.trace_destroy(self.h)
            self.h = C.c_void_p()

    # batch ray queries: intersect!(scene, ray) / intersect_p(scene, ray) over n rays
    def intersect(self, o, d, t_max=None):
        o = np.ascontiguousarray(o, dtype=np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(d, dtype=np.float32).reshape(-1, 3)
        n = len(o)
        t = np.full(n, np.inf, dtype=np.float32) if t_max is None else np.ascontiguousarray(t_max, dtype=np.float32).copy()
        prim = np.zeros(n, dtype=np.uint32)
        b = np.zeros((n, 2), dtype=np.float32)
        self.check(self.lib.trace_intersect(self.h, _lib.ptr(o), _lib.ptr(d), _lib.ptr(t), n, _lib.ptr(prim), _lib.ptr(b)))
        return prim, t, b

    def occluded(self, o, d, t_max=None):
        o = np.ascontiguousarray(o, dtype=np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(d, dtype=np.float32).reshape(-1, 3)
        n = len(o)
        t = np.full(n, np.inf, dtype=np.float32) if t_max is None else np.ascontiguousarray(t_max, dtype=np.float32)
        out = np.zeros(n, dtype=np.uint8)
        self.check(self.lib.trace_occluded(self.h, _lib.ptr(o), _lib.ptr(d), _lib.ptr(t), n, _lib.ptr(out)))
        return out.astype(bool)


def comm_unique_id():
    """128-byte id of a new communicator (rank 0 creates it and hands it to the other ranks out of band)."""
    buf = C.create_string_buffer(_lib.COMM_ID_BYTES)
    rc = _lib.load().trace_comm_unique_id(buf)
    if rc != 0:
        raise RuntimeError(f"trace_comm_unique_id failed ({rc}): libnccl.so.2 could not be loaded")
    return buf.raw


_default_ctx = None


def default_context():
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


def _check_shaded(flat):
    if flat.has_unshaded:
        raise ValueError("every primitive needs a material to be rendered (the reference raises a MethodError for a "
                         "hit without a BSDF, src/integrators/sampler.jl:76-81)")


class WhittedIntegrator:
    """WhittedIntegrator(camera, sampler, max_depth); call it on a Scene (src/integrators/sampler.jl:3-56).
    Accumulates into camera.film.pixels and saves the film, like the reference."""

    def __init__(self, camera, sampler, max_depth, seed=0x5EED0001, context=None):
        self.camera, self.sampler, self.max_depth = camera, sampler, int(max_depth)
        self.seed = seed
        self.context = context

    def __call__(self, scene):
        ctx = self.context or default_context()
        flat = ctx.upload(scene)
        _check_shaded(flat)
        film = self.camera.film
        cam, fd = self.camera.pod(), film.desc()
        ctx.check(ctx.lib.trace_render_whitted(ctx.h, C.byref(cam), C.byref(fd), self.sampler.samples_per_pixel,
                                               self.max_depth, C.c_uint64(self.seed), _lib.ptr(film.pixels)))
        return film.save()


class SPPMIntegrator:
    """SPPMIntegrator(camera, initial_search_radius, max_depth, n_iterations, photons_per_iteration = -1,
    write_frequency = 1); call it on a Scene (src/integrators/sppm.jl:108-173)."""

    def __init__(self, camera, initial_search_radius, max_depth, n_iterations, photons_per_iteration=-1,
                 write_frequency=1, seed=0x5EED0001, context=None):
        self.camera = camera
        self.initial_search_radius = f32(initial_search_radius)
        self.max_depth, self.n_iterations = int(max_depth), int(n_iterations)
        if photons_per_iteration <= 0:                                   # :121-124 (area(crop_bounds), Q22)
            photons_per_iteration = int(camera.film.crop_bounds.area())
        self.photons_per_iteration = int(photons_per_iteration)
        self.write_frequency = int(write_frequency)
        self.seed = seed
        self.context = context

    def __call__(self, scene):
        ctx = self.context or default_context()
        flat = ctx.upload(scene)
        _check_shaded(flat)
        film = self.camera.film
        cam, fd = self.camera.pod(), film.desc()
        h, w = film.pixels.shape[:2]
        rgb = np.zeros((h, w, 3), dtype=np.float32)

        def on_image(_user, iteration, ptr):                             # :167-171
            img = np.ctypeslib.as_array(ptr, shape=(h, w, 3))
            film.set_image(img)
            film.save()

        cb = _lib.SPPM_CB(on_image) if film.filename else C.cast(None, _lib.SPPM_CB)
        ctx.check(ctx.lib.trace_render_sppm(ctx.h, C.byref(cam), C.byref(fd), float(self.initial_search_radius),
                                            self.max_depth, self.n_iterations, self.photons_per_iteration,
                                            self.write_frequency, C.c_uint64(self.seed), cb, None, _lib.ptr(rgb)))
        film.set_image(rgb)
        return film.save()
