"""Host-side mirror of Trace.jl's scene-description API (same names, argument meaning and behaviour):
ShapeCore / Sphere / TriangleMesh / Triangle / create_triangle_mesh (src/shapes/*.jl), GeometricPrimitive
(src/primitive.jl), BVHAccel (src/accel/bvh.jl:50-80), Scene (src/Trace.jl:176-187), materials and textures
(src/materials/material.jl, src/textures/basic.jl), lights (src/lights/point.jl, spot.jl), load_triangle_mesh
(src/model_loader.jl, re-done as a binary-PLY reader).  Everything here is description; traversal and shading run in
libtrace_cuda.so.
"""
import ctypes as C
import struct

import numpy as np

from . import _lib
from .geometry import (Bounds3, Transformation, _deg2rad, _v3, f32)


# ------------------------------------------------------------------ spectrum / textures / materials
class RGBSpectrum:
    __slots__ = ("c",)

    def __init__(self, r=0.0, g=None, b=None):
        self.c = np.array([r, r if g is None else g, r if b is None else b], dtype=np.float32)

    def __mul__(self, f):
        if isinstance(f, RGBSpectrum):
            return RGBSpectrum(*(self.c * f.c))
        return RGBSpectrum(*(self.c * f32(f)))

    __rmul__ = __mul__


class ConstantTexture:
    """src/textures/basic.jl:4-10"""
    __slots__ = ("value",)

    def __init__(self, value):
        self.value = value


class ScaleTexture:
    """src/textures/basic.jl:12-19: texture_1(si) * texture_2(si)."""
    __slots__ = ("texture_1", "texture_2")

    def __init__(self, texture_1, texture_2):
        self.texture_1, self.texture_2 = texture_1, texture_2


class MixTexture:
    """src/textures/basic.jl:21-37: (1 - t) * texture_1(si) + t * texture_2(si) with t = mix(si)::Float32."""
    __slots__ = ("texture_1", "texture_2", "mix")

    def __init__(self, texture_1, texture_2, mix):
        self.texture_1, self.texture_2, self.mix = texture_1, texture_2, mix


def _tex_value(t):
    """Value of a texture tree as the reference evaluates it at a hit.  The leaves the reference can build without a
    2D mapping are ConstantTextures, so Scale / Mix trees do not vary over the surface: they fold, in Float32 and in
    the reference's operation order, into the constant the device material carries (Bilerp / mappings: out of scope)."""
    if isinstance(t, ConstantTexture):
        v = t.value
        return v.c.astype(np.float32) if isinstance(v, RGBSpectrum) else f32(v)
    if isinstance(t, ScaleTexture):
        return (_tex_value(t.texture_1) * _tex_value(t.texture_2)).astype(np.float32)
    if isinstance(t, MixTexture):
        m = _tex_value(t.mix)
        if np.ndim(m) != 0:
            raise TypeError("MixTexture: `mix` must be a Float32 texture (textures/basic.jl:34)")
        m = f32(m)
        return ((f32(1) - m) * _tex_value(t.texture_1) + m * _tex_value(t.texture_2)).astype(np.float32)
    if isinstance(t, RGBSpectrum):
        return t.c.astype(np.float32)
    return f32(t)


def _tex_rgb(t):
    v = _tex_value(t)
    return v if np.ndim(v) else np.full(3, v, dtype=np.float32)


def _tex_f(t):
    v = _tex_value(t)
    if np.ndim(v):
        raise TypeError("a Float32 texture is required here, got a spectrum")
    return f32(v)


class Material:
    def pod(self):
        raise NotImplementedError


class MatteMaterial(Material):
    def __init__(self, Kd, sigma):
        self.Kd, self.sigma = Kd, sigma

    def pod(self):
        return (_lib.MAT_MATTE, _tex_rgb(self.Kd), np.zeros(3, np.float32), 1.0, _tex_f(self.sigma), 0.0, 0)


class MirrorMaterial(Material):
    def __init__(self, Kr):
        self.Kr = Kr

    def pod(self):
        return (_lib.MAT_MIRROR, _tex_rgb(self.Kr), np.zeros(3, np.float32), 1.0, 0.0, 0.0, 0)


class GlassMaterial(Material):
    def __init__(self, Kr, Kt, u_roughness, v_roughness, index, remap_roughness):
        self.Kr, self.Kt, self.u_roughness, self.v_roughness = Kr, Kt, u_roughness, v_roughness
        self.index, self.remap_roughness = index, remap_roughness

    def pod(self):
        return (_lib.MAT_GLASS, _tex_rgb(self.Kr), _tex_rgb(self.Kt), _tex_f(self.index), _tex_f(self.u_roughness),
                _tex_f(self.v_roughness), int(bool(self.remap_roughness)))


class PlasticMaterial(Material):
    def __init__(self, Kd, Ks, roughness, remap_roughness):
        self.Kd, self.Ks, self.roughness, self.remap_roughness = Kd, Ks, roughness, remap_roughness

    def pod(self):
        return (_lib.MAT_PLASTIC, _tex_rgb(self.Kd), _tex_rgb(self.Ks), 1.0, _tex_f(self.roughness), 0.0,
                int(bool(self.remap_roughness)))


# ------------------------------------------------------------------ shapes
class ShapeCore:
    """src/shapes/Shape.jl:1-15"""
    __slots__ = ("object_to_world", "world_to_object", "reverse_orientation", "transform_swaps_handedness")

    def __init__(self, object_to_world, reverse_orientation=False):
        self.object_to_world = object_to_world
        self.world_to_object = object_to_world.inv()
        self.reverse_orientation = bool(reverse_orientation)
        self.transform_swaps_handedness = object_to_world.swaps_handedness()

    @property
    def flip(self):
        return self.reverse_orientation != self.transform_swaps_handedness


def _clampf(x, lo, hi):
    return hi if x > hi else (lo if x < lo else x)


class Sphere:
    """src/shapes/sphere.jl:1-37"""

    def __init__(self, core, radius, *args):
        if len(args) == 1:
            z_min, z_max, phi_max = -f32(radius), f32(radius), args[0]
        else:
            z_min, z_max, phi_max = args
        radius, z_min, z_max, phi_max = f32(radius), f32(z_min), f32(z_max), f32(phi_max)
        self.core = core
        self.radius = radius
        self.z_min = f32(_clampf(min(z_min, z_max), -radius, radius))
        self.z_max = f32(_clampf(max(z_min, z_max), -radius, radius))
        self.theta_min = f32(np.arccos(f32(_clampf(f32(min(z_min, z_max) / radius), f32(-1), f32(1)))))
        self.theta_max = f32(np.arccos(f32(_clampf(f32(max(z_min, z_max) / radius), f32(-1), f32(1)))))
        self.phi_max = _deg2rad(_clampf(phi_max, f32(0), f32(360)))

    def object_bound(self):
        r = self.radius
        return Bounds3([-r, -r, self.z_min], [r, r, self.z_max])

    def world_bound(self):
        return self.core.object_to_world.bounds(self.object_bound())


class TriangleMesh:
    """src/shapes/triangle_mesh.jl:1-30.  `indices` are 1-based like the reference's; vertices are moved to world
    space by the constructor (:23)."""

    def __init__(self, object_to_world, n_triangles, indices, n_vertices, vertices, normals=None, tangents=None, uv=None):
        self.n_triangles = int(n_triangles)
        self.n_vertices = int(n_vertices)
        self.vertices = object_to_world.points(np.asarray(vertices, dtype=np.float32).reshape(-1, 3))
        self.indices = np.asarray(indices, dtype=np.uint32).reshape(-1).copy()
        self.normals = None if normals is None else np.asarray(normals, dtype=np.float32).reshape(-1, 3).copy()
        if tangents is not None or uv is not None:
            raise NotImplementedError("per-vertex tangents / uv are outside the hot-path scope (DESIGN.md)")

    def triangle_vertices(self):
        """[n_triangles, 3, 3] world-space vertex positions."""
        idx = self.indices.reshape(-1, 3).astype(np.int64) - 1
        return self.vertices[idx]

    def triangle_normals(self):
        if self.normals is None:
            return None
        idx = self.indices.reshape(-1, 3).astype(np.int64) - 1
        return self.normals[idx]


class Triangle:
    """src/shapes/triangle_mesh.jl:32-44 (i is the 0-based triangle number here)."""
    __slots__ = ("core", "mesh", "i")

    def __init__(self, core, mesh, i):
        self.core, self.mesh, self.i = core, mesh, int(i)

    def vertices(self):
        idx = self.mesh.indices[3 * self.i:3 * self.i + 3].astype(np.int64) - 1
        return self.mesh.vertices[idx]

    def world_bound(self):
        v = self.vertices()
        return Bounds3(v.min(axis=0), v.max(axis=0))

    def object_bound(self):
        v = self.core.world_to_object.points(self.vertices())
        return Bounds3(v.min(axis=0), v.max(axis=0))

    def area(self):
        v = self.vertices().astype(np.float32)
        c = np.cross(v[1] - v[0], v[2] - v[0]).astype(np.float32)
        return f32(0.5) * f32(np.sqrt(np.sum(c * c, dtype=np.float32)))


def create_triangle_mesh(core, n_triangles, indices, n_vertices, vertices, normals=None, tangents=None, uv=None):
    """src/shapes/triangle_mesh.jl:46-59: returns the list of Triangle shapes."""
    mesh = TriangleMesh(core.object_to_world, n_triangles, indices, n_vertices, vertices, normals, tangents, uv)
    return [Triangle(core, mesh, i) for i in range(mesh.n_triangles)]


def load_triangle_mesh(model_file, core=None):
    """Behaviour of src/model_loader.jl:1-53 for a binary little-endian PLY with x,y,z,nx,ny,nz vertices and
    triangle faces: one mesh, per-vertex normals, 0-based file indices shifted to 1-based (:35), every triangle shares
    `core`.  Returns (triangle_meshes, triangles)."""
    if core is None:
        core = ShapeCore(Transformation(), False)
    with open(model_file, "rb") as fh:
        data = fh.read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    header = data[:end].decode("ascii").split("\n")
    if not any(h.startswith("format binary_little_endian") for h in header):
        raise ValueError("only binary_little_endian PLY is supported")
    n_vert = n_face = 0
    props = []
    cur = None
    for h in header:
        w = h.split()
        if len(w) >= 3 and w[0] == "element":
            cur = w[1]
            if cur == "vertex":
                n_vert = int(w[2])
            elif cur == "face":
                n_face = int(w[2])
        elif len(w) >= 3 and w[0] == "property" and cur == "vertex":
            props.append((w[1], w[2]))
    names = [p[1] for p in props]
    if any(p[0] != "float" for p in props) or names[:3] != ["x", "y", "z"]:
        raise ValueError("unsupported PLY vertex layout")
    vdt = np.dtype([(n, "<f4") for n in names])
    verts = np.frombuffer(data, dtype=vdt, count=n_vert, offset=end)
    off = end + n_vert * vdt.itemsize
    fdt = np.dtype([("n", "u1"), ("i", "<i4", 3)])
    faces = np.frombuffer(data, dtype=fdt, count=n_face, offset=off)
    if not np.all(faces["n"] == 3):
        raise ValueError("only triangles supported")
    pos = np.stack([verts["x"], verts["y"], verts["z"]], axis=1).astype(np.float32)
    nrm = None
    if all(k in names for k in ("nx", "ny", "nz")):
        nrm = np.stack([verts["nx"], verts["ny"], verts["nz"]], axis=1).astype(np.float32)
    indices = (faces["i"].astype(np.int64) + 1).astype(np.uint32).reshape(-1)
    mesh = TriangleMesh(core.object_to_world, n_face, indices, n_vert, pos, nrm)
    return [mesh], TriangleSet(core, mesh)


class TriangleSet:
    """All triangles of one mesh as a single sequence object (avoids 10^6 Python objects); indexing yields Triangle."""

    def __init__(self, core, mesh):
        self.core, self.mesh = core, mesh

    def __len__(self):
        return self.mesh.n_triangles

    def __getitem__(self, i):
        if i < 0 or i >= len(self):
            raise IndexError(i)
        return Triangle(self.core, self.mesh, i)


# ------------------------------------------------------------------ primitives / accel / scene
class GeometricPrimitive:
    """src/primitive.jl:1-10"""
    __slots__ = ("shape", "material")

    def __init__(self, shape, material=None):
        self.shape, self.material = shape, material

    def world_bound(self):
        return self.shape.world_bound()


class PrimitiveBatch:
    """[GeometricPrimitive(t, material) for t in triangles] for a whole TriangleSet, kept as arrays."""

    def __init__(self, triangles, material):
        if not isinstance(triangles, TriangleSet):
            raise TypeError("PrimitiveBatch takes a TriangleSet")
        self.triangles, self.material = triangles, material

    def __len__(self):
        return len(self.triangles)


def _expand(primitives):
    """-> kind[int8], (shape records), bounds[n,6]; keeps the caller's primitive order."""
    items = []     # (kind, payload)
    for p in primitives:
        if isinstance(p, PrimitiveBatch):
            items.append(("batch", p))
        elif isinstance(p, BVHAccel):
            items.append(("bvh", p))
        elif isinstance(p, GeometricPrimitive):
            items.append(("sphere" if isinstance(p.shape, Sphere) else "tri", p))
        else:
            raise TypeError(f"not a primitive: {type(p)}")
    return items


# optional replacement of the native tree build: f(prim_bounds [n,6], max_node_primitives, builder) -> (nodes, order)
BVH_BUILD_HOOK = None


class BVHAccel:
    """BVHAccel(primitives, max_node_primitives = 1), src/accel/bvh.jl:50-80.  The build itself is
    trace_bvh_build in libtrace_cuda.so's host part (the reference's SAH split logic)."""

    def __init__(self, primitives, max_node_primitives=1, builder="reference", device=0):
        """builder = "reference": the reference's split logic, bit-identical tree (src/accel/bvh.jl:55-206).
        builder = "sah": opt-in conventional binned SAH (trace_bvh_build_sah) - same hits, ties aside; less traversal.
        builder = "lbvh": opt-in LBVH built on GPU `device` (trace_bvh_build_gpu) - same hits, ties aside; `device` is
        used by this builder only (multi-rank callers pass their own GPU)."""
        if builder not in ("reference", "sah", "lbvh"):
            raise ValueError("builder must be 'reference', 'sah' or 'lbvh'")
        self.builder = builder
        self.max_node_primitives = min(255, int(max_node_primitives))
        self.items = _expand(primitives)
        # flat per-primitive table in the caller's order
        bounds = []
        self.flat = []          # (kind, ref, local index)
        for kind, p in self.items:
            if kind == "batch":
                tv = p.triangles.mesh.triangle_vertices()
                b = np.concatenate([tv.min(axis=1), tv.max(axis=1)], axis=1).astype(np.float32)
                bounds.append(b)
                self.flat.append((kind, p, len(p)))
            elif kind == "bvh":
                bounds.append(p.world_bound().as6()[None, :])
                self.flat.append((kind, p, 1))
            else:
                bounds.append(p.world_bound().as6()[None, :])
                self.flat.append((kind, p, 1))
        self.n_primitives = int(sum(f[2] for f in self.flat))
        if self.n_primitives == 0:
            self.nodes = np.zeros(0, dtype=_lib.node_dtype)
            self.order = np.zeros(0, dtype=np.uint32)
            return
        self.prim_bounds = np.ascontiguousarray(np.concatenate(bounds, axis=0), dtype=np.float32)
        if BVH_BUILD_HOOK is not None:      # (bench.py --impl reference: the checker's builder, no product library in the process)
            self.nodes, self.order = BVH_BUILD_HOOK(self.prim_bounds, self.max_node_primitives, builder)
            return
        lib = _lib.load()
        h = C.c_void_p()
        if builder == "lbvh":
            rc = lib.trace_bvh_build_gpu(int(device), _lib.ptr(self.prim_bounds), self.n_primitives,
                                         self.max_node_primitives, C.byref(h))
            if rc != 0:
                cause = {5: "NaN bounds", 6: "tree deeper than 64 levels: use builder='sah'",
                         7: f"CUDA error or no CUDA device (device {device}); there is no CPU fallback"}.get(rc, "")
                raise RuntimeError(f"trace_bvh_build_gpu failed ({rc}): {cause}")
        else:
            build = lib.trace_bvh_build if builder == "reference" else lib.trace_bvh_build_sah
            rc = build(_lib.ptr(self.prim_bounds), self.n_primitives, self.max_node_primitives, C.byref(h))
            if rc != 0:
                raise RuntimeError(f"trace_bvh_build failed ({rc})")
        try:
            self.nodes = np.zeros(lib.trace_bvh_num_nodes(h), dtype=_lib.node_dtype)
            self.order = np.zeros(lib.trace_bvh_num_prims(h), dtype=np.uint32)
            lib.trace_bvh_copy(h, _lib.ptr(self.nodes), _lib.ptr(self.order))
        finally:
            lib.trace_bvh_free(h)

    def world_bound(self):
        if len(self.nodes) == 0:
            return Bounds3()
        return Bounds3(self.nodes[0]["bmin"], self.nodes[0]["bmax"])


class PointLight:
    """src/lights/point.jl:1-25"""

    def __init__(self, light_to_world, i):
        self.light_to_world = light_to_world
        self.world_to_light = light_to_world.inv()
        self.i = i
        self.position = light_to_world.point(_v3(0.0))

    def pod(self):
        return (_lib.LIGHT_POINT, self.light_to_world.m, self.light_to_world.inv_m, self.i.c, self.position, 0.0, 0.0)


class SpotLight:
    """src/lights/spot.jl:1-20"""

    def __init__(self, light_to_world, i, total_width, falloff_start):
        self.light_to_world = light_to_world
        self.world_to_light = light_to_world.inv()
        self.i = i
        self.position = light_to_world.point(_v3(0.0))
        self.cos_total_width = f32(np.cos(_deg2rad(total_width)))
        self.cos_falloff_start = f32(np.cos(_deg2rad(falloff_start)))

    def pod(self):
        return (_lib.LIGHT_SPOT, self.light_to_world.m, self.light_to_world.inv_m, self.i.c, self.position,
                self.cos_total_width, self.cos_falloff_start)


class DirectionalLight:
    """src/lights/directional.jl:1-56.  world_radius / world_center stay 0 until preprocess!(light, scene) is called,
    exactly like the reference (Scene's constructor does not do it, src/Trace.jl:184)."""

    def __init__(self, light_to_world, l, direction):
        from .geometry import normalize
        self.light_to_world = light_to_world
        self.world_to_light = light_to_world.inv()
        self.i = l
        self.direction = normalize(light_to_world.vector(direction))
        self.world_radius = f32(0)
        self.world_center = _v3(0.0)

    def preprocess(self, scene):                      # preprocess!, directional.jl:35-37 + bounding_sphere, bounds.jl:145-149
        b = scene.bound
        center = ((b.p_min + b.p_max) / f32(2)).astype(np.float32)
        inside = bool(np.all(center >= b.p_min) and np.all(center <= b.p_max))
        d = center - b.p_max
        self.world_center = center
        self.world_radius = f32(np.sqrt(f32(f32(f32(d[0] * d[0]) + f32(d[1] * d[1])) + f32(d[2] * d[2])))) if inside else f32(0)
        scene._flat = None

    def pod(self):
        return (_lib.LIGHT_DIRECTIONAL, self.light_to_world.m, self.light_to_world.inv_m, self.i.c, self.direction,
                self.world_radius, 0.0)


class Scene:
    """Scene(lights, aggregate), src/Trace.jl:176-187."""

    def __init__(self, lights, aggregate):
        self.lights = list(lights)
        self.aggregate = aggregate
        self.bound = aggregate.world_bound()
        self._flat = None

    def flatten(self):
        if self._flat is None:
            self._flat = FlatScene(self)
        return self._flat


def _is_tensor(a):
    return hasattr(a, "is_cuda") and hasattr(a, "data_ptr")


class DeviceMeshScene:
    """A triangle-only scene whose per-triangle arrays live on the GPU (extension: the reference has no counterpart).
    Context.upload builds its tree (the LBVH of BVHAccel(..., builder="lbvh")) and writes every scene buffer on the
    device (trace_scene_upload_mesh_device): nothing proportional to the triangle count crosses to the host, so
    geometry made on the GPU (simulation output, procedural meshes, a change of topology) is rebuilt without a round
    trip through host memory.  The scene is the one BVHAccel(builder="lbvh") + Scene would give for the same triangles,
    with the triangle index as the primitive index queries report.

      vertices      [n, 3, 3] float32 world space
      materials     list of Material; material_ids [n] integers indexing it (None: all 0)
      normals       [n, 3, 3] float32 or None; applied to the triangles whose flags have TRI_HAS_NORMALS
      flags         [n] uint8 TRI_FLIP | TRI_HAS_NORMALS, or None (all 0)

    Arrays are contiguous CUDA tensors on one device (read in place; the context's device at upload) or numpy arrays,
    which are moved to `device` (default: the tensors' device, else cuda:0) through torch.  Context.upload caches by
    identity: a new DeviceMeshScene triggers a new build; to move the same triangles use Context.refit."""

    def __init__(self, lights, vertices, materials, material_ids=None, normals=None, flags=None, max_node_primitives=1,
                 device=None):
        self.lights = list(lights)
        self.materials = list(materials)
        for m in self.materials:
            if not isinstance(m, Material):
                raise ValueError(f"materials must be Material objects, got {type(m).__name__}")
        self.max_node_primitives = int(max_node_primitives)
        self.has_unshaded = False             # every triangle indexes a material
        n = self._check(vertices, "vertices", None, (3, 3), ("float32",))
        self.n_tris = n
        self._check(normals, "normals", n, (3, 3), ("float32",))
        self._check(flags, "flags", n, (), ("uint8",))
        self._check(material_ids, "material_ids", n, (), ("int8", "int16", "int32", "int64", "uint8", "uint16", "uint32"),
                    tensor_dtypes=("int32", "int64"))
        k = len(self.materials)
        if n > 0 and k == 0:
            raise ValueError("a scene with triangles needs at least one material")
        if isinstance(material_ids, np.ndarray) and n > 0:
            lo, hi = int(material_ids.min()), int(material_ids.max())
            if lo < 0 or hi >= k:
                raise ValueError(f"material_ids must be in [0, {k}), got values in [{lo}, {hi}]")
        given = [a for a in (vertices, normals, flags, material_ids) if _is_tensor(a)]
        devs = {a.device.index for a in given}
        if len(devs) > 1:
            raise ValueError(f"the CUDA tensors are on different devices {sorted(devs)}")
        if device is not None and devs and int(device) not in devs:
            raise ValueError(f"the CUDA tensors are on device {devs.pop()}, not device {int(device)}")
        self.device = int(device) if device is not None else (devs.pop() if devs else 0)
        import torch
        dev = torch.device("cuda", self.device)
        to_dev = lambda a: None if a is None else (a if _is_tensor(a) else torch.from_numpy(np.ascontiguousarray(a)).to(dev))
        self.vertices, self.normals, self.flags = to_dev(vertices), to_dev(normals), to_dev(flags)
        ids = to_dev(material_ids)
        self.material_ids = ids if ids is None or ids.dtype == torch.int32 else ids.to(torch.int32)
        if n == 0:
            self.bound = Bounds3()
        else:                                 # exact: min / max round nothing
            v = self.vertices.view(n * 3, 3)
            lo_hi = torch.stack([v.amin(0), v.amax(0)]).cpu().numpy()
            self.bound = Bounds3(lo_hi[0], lo_hi[1])

    @staticmethod
    def _check(a, what, n, tail, dtypes, tensor_dtypes=None):
        """-> the row count; ValueError on a wrong kind, shape, dtype, layout"""
        if a is None:
            if what == "vertices":
                raise ValueError("vertices are required")
            return n
        if _is_tensor(a):
            if not a.is_cuda:
                raise ValueError(f"{what}: a CPU tensor; pass a CUDA tensor or a numpy array")
            dt = str(a.dtype).replace("torch.", "")
            if dt not in (tensor_dtypes or dtypes):
                raise ValueError(f"{what} must have dtype {' / '.join(tensor_dtypes or dtypes)}, got {dt}")
            if not a.is_contiguous():
                raise ValueError(f"{what} must be contiguous")
            shape = tuple(a.shape)
        elif isinstance(a, np.ndarray):
            if a.dtype.name not in dtypes:
                raise ValueError(f"{what} must have dtype {' / '.join(dtypes) if len(dtypes) < 3 else 'integer'}, got {a.dtype.name}")
            shape = a.shape
        else:
            raise ValueError(f"{what} must be a numpy array or a CUDA tensor, got {type(a).__name__}")
        rows = shape[0] if len(shape) >= 1 else -1
        if len(shape) != 1 + len(tail) or tuple(shape[1:]) != tuple(tail) or (n is not None and rows != n):
            want = ("n" if n is None else str(n),) + tuple(str(t) for t in tail)
            raise ValueError(f"{what} must have shape ({', '.join(want)}{',' if not tail else ''}), got {tuple(shape)}")
        if rows >= 1 << 30:
            raise ValueError(f"{what}: at most 2^30 - 1 triangles")
        return rows

    def desc(self, device):
        """-> (MeshDeviceDesc, the host arrays it points into) for an upload to a context on `device`"""
        if int(device) != self.device:
            raise ValueError(f"the scene's arrays are on device {self.device}, the context is on device {int(device)}")
        mats = np.zeros(max(1, len(self.materials)), dtype=_lib.material_dtype)
        for i, m in enumerate(self.materials):
            mats[i] = m.pod()
        lights = np.zeros(len(self.lights), dtype=_lib.light_dtype)
        for i, l in enumerate(self.lights):
            k, m, im, I, pos, ct, cf = l.pod()
            lights[i] = (k, m.reshape(-1), im.reshape(-1), I, pos, ct, cf)
        ptr = lambda t: None if t is None else t.data_ptr()
        d = _lib.MeshDeviceDesc()
        d.n_tris = self.n_tris
        d.tri_vertices, d.tri_normals = ptr(self.vertices), ptr(self.normals)
        d.tri_flags, d.tri_materials = ptr(self.flags), ptr(self.material_ids)
        d.max_node_primitives = self.max_node_primitives
        d.n_materials, d.materials = len(self.materials), _lib.ptr(mats)
        d.n_lights, d.lights = len(lights), _lib.ptr(lights)
        return d, (mats, lights)


class CompositeScene:
    """A Scene (the environment) with DeviceMeshScenes attached to it (extension: the reference has no counterpart).
    `mesh` is one DeviceMeshScene or an iterable of 1 to 64 of them, the slots in order.  Context.upload uploads
    `scene` once and attaches the meshes on the GPU (trace_scene_attach_meshes_device): each new mesh object rebuilds
    only that mesh's tree, whatever the environment holds (analytic spheres, nested BVHAccels, a reference or sah tree).
    The device scene is the one Scene(lights, BVHAccel) uploads when its root has the environment's tree as first child
    and a balanced tree over the meshes' trees, in slot order, as second: the meshes' triangles come after the
    environment's in slot order (queries report triangle i of mesh j as the environment's primitive count + the
    triangles of meshes 0 .. j - 1 + i), their materials and lights after the environment's.

    Context.upload caches by identity: the environment is uploaded again only when its flattening changed, a slot is
    rebuilt only when it holds a new object.  To move triangles use Context.refit with the vertices of all triangles,
    the environment's first, then the meshes' in slot order.  `mesh` is the mesh when there is exactly one, else None."""

    MAX_MESHES = 64

    def __init__(self, scene, mesh):
        if not isinstance(scene, Scene):
            raise ValueError(f"scene must be a Scene, got {type(scene).__name__}")
        single = isinstance(mesh, DeviceMeshScene)
        try:
            meshes = (mesh,) if single else tuple(mesh)
        except TypeError:
            raise ValueError(f"mesh must be a DeviceMeshScene, got {type(mesh).__name__}") from None
        if not 1 <= len(meshes) <= self.MAX_MESHES:
            raise ValueError(f"meshes: between 1 and {self.MAX_MESHES} DeviceMeshScenes, got {len(meshes)}")
        for j, m in enumerate(meshes):
            if not isinstance(m, DeviceMeshScene):
                raise ValueError(f"mesh must be a DeviceMeshScene, got {type(m).__name__}" + ("" if single else f" (mesh {j})"))
            if m.n_tris == 0:
                raise ValueError("mesh must hold at least one triangle" + ("" if single else f" (mesh {j})"))
        self.scene, self.meshes = scene, meshes
        self.mesh = meshes[0] if len(meshes) == 1 else None
        self.lights = scene.lights + [l for m in meshes for l in m.lights]
        self.bound = scene.bound
        for m in meshes:
            self.bound = self.bound.union(m.bound)

    @property
    def has_unshaded(self):
        return self.scene.flatten().has_unshaded


class FlatScene:
    """The POD upload (trace_scene_desc): BVH nodes with nested BVHAccel primitives spliced in place, the BVH-ordered
    primitive list, triangle / sphere arrays, materials and lights."""

    def __init__(self, scene):
        self.materials = []
        self._mat_ids = {}
        self.has_unshaded = False
        tri_v, tri_n, tri_f = [], [], []
        spheres = []
        self.n_tris = 0
        self._orig = 0
        self.tri_sources = []       # where the triangles come from, in triangle order: a batch's mesh or one Triangle
        self.sphere_bounds = []     # world_bound() of each sphere (the bounds its tree was built with)
        self.stale = False          # Context.refit moved the vertices on the device: nodes / tri_vertices are old
        nodes, prims = self._flatten_bvh(scene.aggregate, tri_v, tri_n, tri_f, spheres)
        self.nodes = nodes
        self.prims = prims
        if tri_v:
            self.tri_vertices = np.ascontiguousarray(np.concatenate(tri_v, axis=0), dtype=np.float32)
            self.tri_normals = np.ascontiguousarray(np.concatenate(tri_n, axis=0), dtype=np.float32)
            self.tri_flags = np.ascontiguousarray(np.concatenate(tri_f, axis=0), dtype=np.uint8)
        else:
            self.tri_vertices = np.zeros((0, 3, 3), np.float32)
            self.tri_normals = np.zeros((0, 3, 3), np.float32)
            self.tri_flags = np.zeros(0, np.uint8)
        self.spheres = np.array(spheres, dtype=_lib.sphere_dtype) if spheres else np.zeros(0, _lib.sphere_dtype)
        self.sphere_bounds = np.array(self.sphere_bounds, dtype=np.float32).reshape(-1, 6)
        mats = np.zeros(max(1, len(self.materials)), dtype=_lib.material_dtype)
        for i, m in enumerate(self.materials):
            mats[i] = m.pod()
        self.materials_pod = mats
        self.n_materials = len(self.materials)
        lights = np.zeros(len(scene.lights), dtype=_lib.light_dtype)
        for i, l in enumerate(scene.lights):
            k, m, im, I, pos, ct, cf = l.pod()
            lights[i] = (k, m.reshape(-1), im.reshape(-1), I, pos, ct, cf)
        self.lights = lights

    def _material_id(self, m):
        if m is None:
            # allowed for ray queries (test/test_intersection.jl builds GeometricPrimitive(sphere) without one);
            # the integrators refuse such scenes (the reference raises a MethodError, integrators/sampler.jl:76-81)
            self.has_unshaded = True
            return 0xFFFFFFFF
        k = id(m)
        if k not in self._mat_ids:
            self._mat_ids[k] = len(self.materials)
            self.materials.append(m)
        return self._mat_ids[k]

    def _flatten_bvh(self, bvh, tri_v, tri_n, tri_f, spheres):
        # 1. register shapes of this BVH (caller's order) and build the per-primitive table
        kinds = np.zeros(bvh.n_primitives, dtype=np.uint32)
        index = np.zeros(bvh.n_primitives, dtype=np.uint32)
        mat = np.zeros(bvh.n_primitives, dtype=np.uint32)
        orig = np.zeros(bvh.n_primitives, dtype=np.uint32)
        nested = {}
        pos = 0
        for kind, p, cnt in bvh.flat:
            if kind == "batch":
                mesh, core = p.triangles.mesh, p.triangles.core
                tv = mesh.triangle_vertices()
                tn = mesh.triangle_normals()
                flags = (1 if core.flip else 0) | (2 if tn is not None else 0)
                tri_v.append(tv)
                tri_n.append(tn if tn is not None else np.zeros_like(tv))
                tri_f.append(np.full(cnt, flags, dtype=np.uint8))
                self.tri_sources.append(mesh)
                kinds[pos:pos + cnt] = _lib.PRIM_TRIANGLE
                index[pos:pos + cnt] = np.arange(self.n_tris, self.n_tris + cnt, dtype=np.uint32)
                mat[pos:pos + cnt] = self._material_id(p.material)
                orig[pos:pos + cnt] = np.arange(self._orig, self._orig + cnt, dtype=np.uint32)
                self.n_tris += cnt
                self._orig += cnt
            elif kind == "tri":
                t = p.shape
                tv = t.vertices()[None]
                idx = t.mesh.indices[3 * t.i:3 * t.i + 3].astype(np.int64) - 1
                has_n = t.mesh.normals is not None
                tri_v.append(tv)
                tri_n.append(t.mesh.normals[idx][None] if has_n else np.zeros_like(tv))
                tri_f.append(np.array([(1 if t.core.flip else 0) | (2 if has_n else 0)], dtype=np.uint8))
                self.tri_sources.append(t)
                kinds[pos] = _lib.PRIM_TRIANGLE
                index[pos] = self.n_tris
                mat[pos] = self._material_id(p.material)
                orig[pos] = self._orig
                self.n_tris += 1
                self._orig += 1
            elif kind == "sphere":
                s = p.shape
                o2w = s.core.object_to_world
                spheres.append((o2w.m.reshape(-1), o2w.inv_m.reshape(-1), s.radius, s.z_min, s.z_max, s.theta_min,
                                s.theta_max, s.phi_max, 1 if s.core.flip else 0, 0))
                self.sphere_bounds.append(s.world_bound().as6())
                kinds[pos] = _lib.PRIM_SPHERE
                index[pos] = len(spheres) - 1
                mat[pos] = self._material_id(p.material)
                orig[pos] = self._orig
                self._orig += 1
            else:
                nested[pos] = p
                kinds[pos] = 0xFFFFFFFF
            pos += cnt
        order = bvh.order.astype(np.int64)
        if not nested:
            prims = np.zeros(len(order), dtype=_lib.prim_dtype)
            prims["kind"], prims["index"], prims["material"], prims["original"] = kinds[order], index[order], mat[order], orig[order]
            return bvh.nodes.copy(), prims
        # 2. nested BVHAccel primitives (test/test_intersection.jl:137-138): splice each one's node array in place of
        #    the leaf that holds it; same box tests in the same order as the reference's recursive call.
        out_nodes, out_prims = [], []
        sub = {k: self._flatten_bvh(v, tri_v, tri_n, tri_f, spheres) for k, v in nested.items()}

        def emit(nodes, prim_rows, i, prim_base):
            nd = nodes[i]
            slot = len(out_nodes)
            if (int(nd["meta"]) >> 30) == 3:
                n = int(nd["meta"]) & 0x3FFFFFFF
                off = int(nd["offset"])
                rows = prim_rows[off:off + n]
                if any(r is not None and r[0] == "nested" for r in rows):
                    if n != 1:
                        raise NotImplementedError("a leaf mixing a nested BVHAccel with other primitives")
                    sn, sp = sub[rows[0][1]]
                    emit(sn, [("prim", sp[j]) for j in range(len(sp))], 0, 0)
                    return
                out_nodes.append((nd["bmin"].copy(), nd["bmax"].copy(), len(out_prims), int(nd["meta"])))
                for r in rows:
                    out_prims.append(r[1])
                return
            out_nodes.append(None)
            emit(nodes, prim_rows, i + 1, prim_base)
            second = len(out_nodes)
            emit(nodes, prim_rows, int(nd["offset"]), prim_base)
            out_nodes[slot] = (nd["bmin"].copy(), nd["bmax"].copy(), second, int(nd["meta"]))

        rows = []
        for j in order:
            if int(j) in nested:
                rows.append(("nested", int(j)))
            else:
                rows.append(("prim", (kinds[j], index[j], mat[j], orig[j])))
        emit(bvh.nodes, rows, 0, 0)
        nodes = np.zeros(len(out_nodes), dtype=_lib.node_dtype)
        for i, (lo, hi, off, meta) in enumerate(out_nodes):
            nodes[i] = (lo, hi, off, meta)
        prims = np.zeros(len(out_prims), dtype=_lib.prim_dtype)
        for i, r in enumerate(out_prims):
            prims[i] = tuple(int(x) for x in r)
        return nodes, prims

    def gather_vertices(self):
        """[n_tris, 3, 3] float32: the current world-space vertices of the meshes this scene was flattened from, in the
        order of `tri_vertices` (what Context.refit(scene) uploads after the caller moved mesh vertices)."""
        if not self.tri_sources:
            return np.zeros((0, 3, 3), np.float32)
        parts = [src.triangle_vertices() if isinstance(src, TriangleMesh) else src.vertices()[None] for src in self.tri_sources]
        return np.ascontiguousarray(np.concatenate(parts, axis=0), dtype=np.float32)

    def desc(self):
        d = _lib.SceneDesc()
        d.n_nodes, d.nodes = len(self.nodes), _lib.ptr(self.nodes)
        d.n_prims, d.prims = len(self.prims), _lib.ptr(self.prims)
        d.n_tris = len(self.tri_vertices)
        d.tri_vertices = _lib.ptr(self.tri_vertices)
        d.tri_normals = _lib.ptr(self.tri_normals)
        d.tri_flags = _lib.ptr(self.tri_flags)
        d.n_spheres, d.spheres = len(self.spheres), _lib.ptr(self.spheres)
        d.n_materials, d.materials = self.n_materials, _lib.ptr(self.materials_pod)
        d.n_lights, d.lights = len(self.lights), _lib.ptr(self.lights)
        return d
