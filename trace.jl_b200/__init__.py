"""trace.jl_b200 — B200 (sm_100a) backend for Trace.jl's ray-tracing hot path, behind Trace.jl's own API names.

Usage mirrors the reference's scene scripts (docs/code/*.jl):

    import trace_jl_b200 as Trace
    bvh = Trace.BVHAccel(primitives, 1)
    scene = Trace.Scene(lights, bvh)
    Trace.SPPMIntegrator(camera, 0.025, 5, 100)(scene)

Traversal, shading, film accumulation and the SPPM passes run in csrc/libtrace_cuda.so (hand-written CUDA for sm_100a)
through the C ABI in include/trace_cuda.h.  There is no CPU fallback.
"""
from .geometry import (Bounds2, Bounds3, Normal3f, Point2f, Point3f, Transformation, Vec3f, coordinate_system, cross, dot,
                       look_at, norm, normalize, perspective, rotate_x, rotate_y, rotate_z, scale, translate)
from .scene import (BVHAccel, ConstantTexture, MixTexture, ScaleTexture, DeviceMeshScene, DirectionalLight, FlatScene, GeometricPrimitive, GlassMaterial, MatteMaterial, MirrorMaterial,
                    PlasticMaterial, PointLight, PrimitiveBatch, RGBSpectrum, Scene, ShapeCore, Sphere, SpotLight, Triangle,
                    TriangleMesh, TriangleSet, create_triangle_mesh, load_triangle_mesh)
from .render import (Context, comm_unique_id, Film, LanczosSincFilter, PerspectiveCamera, SPPMIntegrator, UniformSampler, WhittedIntegrator,
                     default_context, write_png)
from . import scenes  # noqa: E402
