# TraceCUDA.jl — the reference-side binding a Trace.jl maintainer would add to use libtrace_cuda.so as the GPU backend.
#
# NOT RUNNABLE IN THIS IMAGE (no julia binary); it documents, in the reference's own language, exactly which calls the
# C ABI (include/trace_cuda.h) replaces.  The Python package trace.jl_b200/ is the runnable mirror of this file.
#
#   using Trace, TraceCUDA
#   scene |> TraceCUDA.gpu(Trace.SPPMIntegrator(camera, 0.025f0, 5, 100))      # instead of  scene |> integrator
#   scene |> TraceCUDA.gpu(integrator, TraceCUDA.MultiContext(0:7))            # all eight GPUs of the box (julia -t 8)
#
module TraceCUDA

using Trace
using GeometryBasics

const LIB = get(ENV, "TRACE_CUDA_LIB", "libtrace_cuda.so")

# ---- POD mirrors of include/trace_cuda.h --------------------------------------------------------------------------
struct BVHNode            # trace_bvh_node, 32 B
    bmin::NTuple{3,Float32}
    bmax::NTuple{3,Float32}
    offset::UInt32
    meta::UInt32
end
struct Prim               # trace_prim
    kind::UInt32
    index::UInt32
    material::UInt32
    original::UInt32
end
struct SphereP            # trace_sphere
    m::NTuple{16,Float32}
    inv_m::NTuple{16,Float32}
    radius::Float32; z_min::Float32; z_max::Float32; θ_min::Float32; θ_max::Float32; ϕ_max::Float32
    flip::UInt32; pad::UInt32
end
struct MaterialP          # trace_material
    kind::UInt32
    a::NTuple{3,Float32}; b::NTuple{3,Float32}
    η::Float32; rough_u::Float32; rough_v::Float32
    remap::UInt32
end
struct LightP             # trace_light
    kind::UInt32
    m::NTuple{16,Float32}; inv_m::NTuple{16,Float32}
    i::NTuple{3,Float32}; position::NTuple{3,Float32}
    cos_total_width::Float32; cos_falloff_start::Float32
end
struct SceneDesc          # trace_scene_desc
    n_nodes::Int64; nodes::Ptr{BVHNode}
    n_prims::Int64; prims::Ptr{Prim}
    n_tris::Int64; tri_vertices::Ptr{Float32}; tri_normals::Ptr{Float32}; tri_flags::Ptr{UInt8}
    n_spheres::Int64; spheres::Ptr{SphereP}
    n_materials::Int64; materials::Ptr{MaterialP}
    n_lights::Int64; lights::Ptr{LightP}
end
struct CameraP            # trace_camera
    raster_to_camera::NTuple{16,Float32}
    camera_to_world::NTuple{16,Float32}
    lens_radius::Float32; focal_distance::Float32; shutter_open::Float32; shutter_close::Float32
end
struct FilmP              # trace_film_desc
    crop::NTuple{4,Int32}
    filter_radius::NTuple{2,Float32}
    filter_table::NTuple{256,Float32}
    scale::Float32
end

rowmajor(m::Mat4f) = ntuple(k -> m[(k - 1) ÷ 4 + 1, (k - 1) % 4 + 1], 16)

# ---- context ------------------------------------------------------------------------------------------------------
mutable struct Context
    h::Ptr{Cvoid}
    lock::ReentrantLock
    seed::UInt64            # renders draw seed, seed + 1, ...: a fixed seed makes Julia-side renders reproducible
    function Context(device::Integer = 0; seed::Integer = 0x5EED0001)
        out = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall((:trace_create, LIB), Cint, (Ref{Ptr{Cvoid}}, Cint, Ptr{Cvoid}), out, device, C_NULL)
        rc == 0 || error("trace_create failed ($rc): no CUDA device (there is no CPU fallback)")
        ctx = new(out[], ReentrantLock(), UInt64(seed))
        finalizer(c -> ccall((:trace_destroy, LIB), Cvoid, (Ptr{Cvoid},), c.h), ctx)
    end
end
check(ctx, rc) = rc == 0 || error(unsafe_string(ccall((:trace_last_error, LIB), Cstring, (Ptr{Cvoid},), ctx.h)))
set_option!(ctx::Context, key::AbstractString, v::Integer) =
    check(ctx, ccall((:trace_set_option, LIB), Cint, (Ptr{Cvoid}, Cstring, Int64), ctx.h, key, v))
next_seed!(ctx::Context) = (s = ctx.seed; ctx.seed += 1; s)

# ---- several GPUs of one box: one Context per device, one Julia task per Context ------------------------------------------
# The reference parallelises with Threads.@threads over tiles / photons into shared arrays; across GPUs the library runs
# the two exchange steps itself on NCCL (trace_comm_init).  Here: one process, `Threads.@spawn` per device, all ranks share
# the id through a captured variable, and - film_mode 1 - every GPU writes ITS band of the one shared host film.
struct MultiContext
    ctxs::Vector{Context}
end
function MultiContext(devices::AbstractVector{<:Integer}; seed::Integer = 0x5EED0001)
    ctxs = [Context(d; seed = seed) for d in devices]          # the same seed on every rank: ranks must agree on it
    id = zeros(UInt8, 128)                                      # TRACE_COMM_ID_BYTES
    ccall((:trace_comm_unique_id, LIB), Cint, (Ptr{UInt8},), id) == 0 || error("libnccl.so.2 could not be loaded")
    world = length(ctxs)
    @sync for (r, c) in enumerate(ctxs)                         # trace_comm_init is collective: all ranks concurrently
        Threads.@spawn check(c, ccall((:trace_comm_init, LIB), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Cint, Cint), c.h, id, r - 1, world))
    end
    foreach(c -> set_option!(c, "film_mode", 1), ctxs)
    MultiContext(ctxs)
end
# run f(ctx) on every rank concurrently (every rank must make the same sequence of render calls)
on_all(f, m::MultiContext) = @sync for c in m.ctxs
    Threads.@spawn f(c)
end

# ---- flattening Trace.Scene -> SceneDesc (what trace.jl_b200/scene.py:FlatScene does) -------------------------------
# BVHAccel.nodes are already the reference's LinearBVH array (1-based); convert to 0-based trace_bvh_node.
function flatten_nodes(bvh::Trace.BVHAccel)
    map(bvh.nodes) do n
        if n isa Trace.LinearBVHLeaf
            BVHNode(Tuple(n.bounds.p_min), Tuple(n.bounds.p_max), n.primitives_offset - 1, 0xC0000000 | n.n_primitives)
        else
            BVHNode(Tuple(n.bounds.p_min), Tuple(n.bounds.p_max), n.second_child_offset - 1, UInt32(n.split_axis - 1) << 30)
        end
    end
end

# constants of include/trace_cuda.h
const PRIM_TRIANGLE, PRIM_SPHERE = UInt32(0), UInt32(1)
const MAT_MATTE, MAT_MIRROR, MAT_GLASS, MAT_PLASTIC = UInt32(0), UInt32(1), UInt32(2), UInt32(3)
const LIGHT_POINT, LIGHT_SPOT, LIGHT_DIRECTIONAL = UInt32(0), UInt32(1), UInt32(2)
const NO_MATERIAL = 0xFFFFFFFF

# Textures: the leaves the reference can build without a 2D mapping are constant, so Scale / Mix trees do not vary over the
# surface; they fold here (Float32, the operation order of src/textures/basic.jl:17-36) into the constant the device
# material carries.  BilerpTexture needs a mapping and is not supported.
texval(t::Trace.ConstantTexture) = t.value
texval(t::Trace.ScaleTexture) = texval(t.texture_1) * texval(t.texture_2)
function texval(t::Trace.MixTexture)
    m::Float32 = texval(t.mix)
    (1 - m) * texval(t.texture_1) + m * texval(t.texture_2)
end
texval(t) = error("TraceCUDA: only Constant / Scale / Mix textures are supported on the GPU path, got $(typeof(t))")
rgb3(s::Trace.RGBSpectrum) = (s.c[1], s.c[2], s.c[3])
const ZERO3 = (0f0, 0f0, 0f0)

material_pod(m::Trace.MatteMaterial) = MaterialP(MAT_MATTE, rgb3(texval(m.Kd)), ZERO3, 1f0, Float32(texval(m.σ)), 0f0, 0)
material_pod(m::Trace.MirrorMaterial) = MaterialP(MAT_MIRROR, rgb3(texval(m.Kr)), ZERO3, 1f0, 0f0, 0f0, 0)
material_pod(m::Trace.GlassMaterial) = MaterialP(MAT_GLASS, rgb3(texval(m.Kr)), rgb3(texval(m.Kt)), Float32(texval(m.index)),
    Float32(texval(m.u_roughness)), Float32(texval(m.v_roughness)), UInt32(m.remap_roughness))
material_pod(m::Trace.PlasticMaterial) = MaterialP(MAT_PLASTIC, rgb3(texval(m.Kd)), rgb3(texval(m.Ks)), 1f0,
    Float32(texval(m.roughness)), 0f0, UInt32(m.remap_roughness))

light_pod(l::Trace.PointLight) = LightP(LIGHT_POINT, rowmajor(l.light_to_world.m), rowmajor(l.light_to_world.inv_m),
    rgb3(l.i), Tuple(l.position), 0f0, 0f0)
light_pod(l::Trace.SpotLight) = LightP(LIGHT_SPOT, rowmajor(l.light_to_world.m), rowmajor(l.light_to_world.inv_m),
    rgb3(l.i), Tuple(l.position), l.cos_total_width, l.cos_falloff_start)
# DirectionalLight: `position` carries the direction, `cos_total_width` the world radius (0 until preprocess!, as in the reference)
light_pod(l::Trace.DirectionalLight) = LightP(LIGHT_DIRECTIONAL, rowmajor(l.light_to_world.m), rowmajor(l.light_to_world.inv_m),
    rgb3(l.i), Tuple(l.direction), l.world_radius, 0f0)

flips(core::Trace.ShapeCore) = core.reverse_orientation != core.transform_swaps_handedness

# Everything trace_scene_upload needs, as Julia arrays kept alive by the caller (GC.@preserve) during the ccall.
mutable struct FlatScene
    nodes::Vector{BVHNode}
    prims::Vector{Prim}
    tri_vertices::Vector{Float32}      # [n_tris][3][3], world space
    tri_normals::Vector{Float32}       # [n_tris][3][3]
    tri_flags::Vector{UInt8}           # bit 0: flip orientation, bit 1: has per-vertex normals
    spheres::Vector{SphereP}
    materials::Vector{MaterialP}
    lights::Vector{LightP}
    material_ids::IdDict{Any,UInt32}
    n_original::UInt32                 # running "caller's order" primitive number
    triangles::Vector{Any}             # the Trace.Triangle behind each tri_vertices entry (refit! gathers from them)
    sphere_bounds::Vector{Float32}     # [n_spheres][6] world bounds the tree was built with
end
FlatScene() = FlatScene(BVHNode[], Prim[], Float32[], Float32[], UInt8[], SphereP[], MaterialP[], LightP[], IdDict{Any,UInt32}(), 0,
                        Any[], Float32[])

function material_id!(fs::FlatScene, m)
    m === nothing && return NO_MATERIAL          # fine for intersect!/intersect_p; the integrators refuse such scenes
    get!(fs.material_ids, m) do
        push!(fs.materials, material_pod(m))
        UInt32(length(fs.materials) - 1)
    end
end

# one reference primitive -> one trace_prim row (shape data appended to the shape tables)
function prim_row!(fs::FlatScene, p::Trace.GeometricPrimitive{Trace.Triangle})
    t = p.shape
    ids = t.mesh.indices[t.i:t.i + 2]
    for k in ids
        append!(fs.tri_vertices, Float32.(Tuple(t.mesh.vertices[k])))
    end
    has_n = t.mesh.normals !== nothing
    for k in ids
        append!(fs.tri_normals, has_n ? Float32.(Tuple(t.mesh.normals[k])) : ZERO3)
    end
    push!(fs.tri_flags, UInt8(flips(t.core)) | (UInt8(has_n) << 1))
    push!(fs.triangles, t)
    row = Prim(PRIM_TRIANGLE, UInt32(length(fs.tri_flags) - 1), material_id!(fs, p.material), fs.n_original)
    fs.n_original += 1
    row
end
function prim_row!(fs::FlatScene, p::Trace.GeometricPrimitive{Trace.Sphere})
    s = p.shape
    push!(fs.spheres, SphereP(rowmajor(s.core.object_to_world.m), rowmajor(s.core.object_to_world.inv_m), s.radius,
                              s.z_min, s.z_max, s.θ_min, s.θ_max, s.ϕ_max, UInt32(flips(s.core)), 0))
    b = Trace.world_bound(s)
    append!(fs.sphere_bounds, Float32.((b.p_min..., b.p_max...)))
    row = Prim(PRIM_SPHERE, UInt32(length(fs.spheres) - 1), material_id!(fs, p.material), fs.n_original)
    fs.n_original += 1
    row
end

# Emits bvh's LinearBVH array (preorder, first child = parent + 1) into fs.nodes / fs.prims, 0-based.  A BVHAccel used as
# a primitive (test/test_intersection.jl:137-138) is spliced in place of the leaf that holds it, so the device walks
# the same boxes in the same order as the reference's recursive intersect!.
function emit!(fs::FlatScene, bvh::Trace.BVHAccel, i::Int = 1)
    n = bvh.nodes[i]
    if n isa Trace.LinearBVHLeaf
        held = bvh.primitives[n.primitives_offset:n.primitives_offset + n.n_primitives - 1]
        if any(p -> p isa Trace.BVHAccel, held)
            length(held) == 1 || error("TraceCUDA: a leaf mixing a nested BVHAccel with other primitives")
            return emit!(fs, held[1], 1)
        end
        push!(fs.nodes, BVHNode(Tuple(n.bounds.p_min), Tuple(n.bounds.p_max), UInt32(length(fs.prims)), 0xC0000000 | n.n_primitives))
        for p in held
            push!(fs.prims, prim_row!(fs, p))
        end
    else
        slot = length(fs.nodes) + 1
        push!(fs.nodes, BVHNode(Tuple(n.bounds.p_min), Tuple(n.bounds.p_max), 0, UInt32(n.split_axis - 1) << 30))
        emit!(fs, bvh, i + 1)
        second = UInt32(length(fs.nodes))                       # 0-based index of the node emitted next
        emit!(fs, bvh, Int(n.second_child_offset))
        fs.nodes[slot] = BVHNode(fs.nodes[slot].bmin, fs.nodes[slot].bmax, second, fs.nodes[slot].meta)
    end
    nothing
end
# `original` (what trace_intersect reports, + 1) numbers the primitives in emission order.  Leaves are emitted in
# preorder and the reference's build appends primitives to `bvh.primitives` in that same order (`ordered_primitives`, bvh.jl:97-104), so for
# a BVHAccel without nested accelerators `original + 1` indexes `bvh.primitives` directly.  (The Python mirror still has
# the Vector the caller handed to BVHAccel and numbers in that order instead.)

function flatten(scene::Trace.Scene)
    fs = FlatScene()
    isempty(scene.aggregate.nodes) || emit!(fs, scene.aggregate)
    append!(fs.lights, light_pod.(scene.lights))
    fs
end

const UPLOADED = IdDict{Any,Tuple{Any,FlatScene}}()     # per context: the scene that is on the device + its flattening

function upload!(ctx::Context, scene::Trace.Scene)
    haskey(UPLOADED, ctx) && UPLOADED[ctx][1] === scene && return nothing      # already there (scenes are immutable)
    fs = flatten(scene)
    desc = SceneDesc(length(fs.nodes), pointer(fs.nodes), length(fs.prims), pointer(fs.prims),
                     length(fs.tri_flags), pointer(fs.tri_vertices), pointer(fs.tri_normals), pointer(fs.tri_flags),
                     length(fs.spheres), pointer(fs.spheres), length(fs.materials), pointer(fs.materials),
                     length(fs.lights), pointer(fs.lights))
    GC.@preserve fs check(ctx, ccall((:trace_scene_upload, LIB), Cint, (Ptr{Cvoid}, Ref{SceneDesc}), ctx.h, desc))
    UPLOADED[ctx] = (scene, fs)
    nothing
end

# Animation: move the vertices of the scene's meshes (mesh.vertices[k] = ...), then refit!(ctx, scene) instead of
# building a new BVHAccel.  The tree's topology stays; the library recomputes every box on the GPU (trace_scene_refit).
# Every context that holds the scene (one per GPU) is refit with the same vertices.  A deformation computed on the GPU
# can skip the gather and pass a device buffer to trace_scene_refit_device instead.
function refit!(ctx::Context, scene::Trace.Scene)
    haskey(UPLOADED, ctx) && UPLOADED[ctx][1] === scene || error("TraceCUDA.refit!: this scene is not the one uploaded to ctx")
    fs = UPLOADED[ctx][2]
    v = Vector{Float32}(undef, 9 * length(fs.triangles))
    for (j, t) in enumerate(fs.triangles), (c, k) in enumerate(t.mesh.indices[t.i:t.i + 2])
        v[9 * (j - 1) + 3 * (c - 1) .+ (1:3)] .= Float32.(Tuple(t.mesh.vertices[k]))
    end
    GC.@preserve v fs check(ctx, ccall((:trace_scene_refit, LIB), Cint,
        (Ptr{Cvoid}, Int64, Ptr{Float32}, Ptr{Float32}, Int64, Ptr{Float32}),
        ctx.h, length(fs.triangles), v, C_NULL, length(fs.spheres), isempty(fs.spheres) ? C_NULL : pointer(fs.sphere_bounds)))
    nothing
end

# Geometry made on the GPU (CUDA.jl arrays of a simulation, a procedural mesh, a change of topology): upload it without a
# round trip through host memory.  The library builds the LBVH and packs every scene buffer on the device
# (trace_scene_upload_mesh_device); the scene is the one BVHAccel(builder="lbvh") + Scene would give, with the triangle
# index as the primitive index.  Pointers are raw device addresses on ctx's GPU (e.g. UInt(pointer(cu_array))), read on
# the context's stream: synchronise the work that wrote them first.  `materials` / `lights` are host pods
# (material_pod / light_pod).  Returns the node count; refit! does not apply (call trace_scene_refit_device directly).
struct MeshDeviceDesc
    n_tris::Int64
    tri_vertices::UInt          # device Float32 [9, n_tris] (x y z of p0 p1 p2 per triangle)
    tri_normals::UInt           # same layout, or 0
    tri_flags::UInt             # device UInt8 [n_tris] (bit 0 flip, bit 1 has normals), or 0
    tri_materials::UInt         # device UInt32 [n_tris], 0-based into materials, or 0 (all 0)
    max_node_primitives::Int32
    pad::Int32
    n_materials::Int64; materials::Ptr{Cvoid}
    n_lights::Int64; lights::Ptr{Cvoid}
end
function upload_mesh_device!(ctx::Context, n_tris, vertices, normals, flags, material_ids, materials::Vector, lights::Vector;
                             max_node_primitives = 1)
    GC.@preserve materials lights begin
        d = MeshDeviceDesc(n_tris, UInt(vertices), UInt(normals), UInt(flags), UInt(material_ids), Int32(max_node_primitives),
                           Int32(0), length(materials), pointer(materials), length(lights), pointer(lights))
        n_nodes = Ref{Int64}(0)
        check(ctx, ccall((:trace_scene_upload_mesh_device, LIB), Cint, (Ptr{Cvoid}, Ref{MeshDeviceDesc}, Ref{Int64}),
                         ctx.h, d, n_nodes))
    end
    delete!(UPLOADED, ctx)         # the uploaded scene is no Trace.Scene of this shim
    n_nodes[]
end

# ---- the two functors ------------------------------------------------------------------------------------------------
struct GPU{I<:Trace.Integrator,C}
    integrator::I
    ctx::C                 # Context (one GPU) or MultiContext (several GPUs of the box)
end
gpu(i::Trace.Integrator, ctx = Context()) = GPU(i, ctx)

camera_pod(c::Trace.PerspectiveCamera) = CameraP(
    rowmajor(c.core.raster_to_camera.m), rowmajor(c.core.core.camera_to_world.m),
    c.core.lens_radius, c.core.focal_distance, c.core.core.shutter_open, c.core.core.shutter_close)

function film_pod(f::Trace.Film)
    FilmP(Int32.((f.crop_bounds.p_min..., f.crop_bounds.p_max...)), Tuple(f.filter.radius),
          ntuple(k -> f.filter_table[(k - 1) ÷ 16 + 1, (k - 1) % 16 + 1], 256), f.scale)
end

# (i::SamplerIntegrator)(scene)  — src/integrators/sampler.jl:12-56
function render_whitted!(ctx::Context, i, scene, film, buf)
    lock(ctx.lock) do
        upload!(ctx, scene)
        GC.@preserve buf check(ctx, ccall((:trace_render_whitted, LIB), Cint,
            (Ptr{Cvoid}, Ref{CameraP}, Ref{FilmP}, Cint, Cint, UInt64, Ptr{Float32}),
            ctx.h, camera_pod(i.camera), film_pod(film), i.sampler.samples_per_pixel, i.max_depth, next_seed!(ctx), buf))
    end
end
function (g::GPU{Trace.WhittedIntegrator})(scene::Trace.Scene)
    i = g.integrator
    film = Trace.get_film(i.camera)
    H, W = size(film.pixels)
    buf = zeros(Float32, 4, W, H)                       # row-major [y][x][4] on the C side
    for y in 1:H, x in 1:W
        p = film.pixels[y, x]
        buf[1:3, x, y] .= p.xyz; buf[4, x, y] = p.filter_weight_sum
    end
    if g.ctx isa MultiContext
        # every rank renders its tiles; the library sums the films and every GPU uploads / merges / downloads its own band
        # of `buf` (film_mode 1), so the bands travel over as many PCIe links as there are GPUs
        on_all(c -> render_whitted!(c, i, scene, film, buf), g.ctx)
    else
        render_whitted!(g.ctx, i, scene, film, buf)
    end
    for y in 1:H, x in 1:W
        film.pixels[y, x].xyz = Point3f(buf[1:3, x, y]); film.pixels[y, x].filter_weight_sum = buf[4, x, y]
    end
    Trace.save(film)
end

# (i::SPPMIntegrator)(scene)  — src/integrators/sppm.jl:132-173
function (g::GPU{Trace.SPPMIntegrator,MultiContext})(scene::Trace.Scene)
    # camera paths by image rows, photons by index range; the all-gather of the visible points and the all-reduce of
    # (Phi, M) run inside trace_render_sppm.  Every rank returns the whole image; rank 0's drives the film / PNG writes.
    i = g.integrator
    film = Trace.get_film(i.camera)
    H, W = size(film.pixels)
    images = [zeros(Float32, 3, W, H) for _ in g.ctx.ctxs]
    @sync for (r, c) in enumerate(g.ctx.ctxs)
        Threads.@spawn lock(c.lock) do
            upload!(c, scene)
            GC.@preserve images check(c, ccall((:trace_render_sppm, LIB), Cint,
                (Ptr{Cvoid}, Ref{CameraP}, Ref{FilmP}, Cfloat, Cint, Cint, Int64, Cint, UInt64, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float32}),
                c.h, camera_pod(i.camera), film_pod(film), i.initial_search_radius, i.max_depth, i.n_iterations,
                i.photons_per_iteration, 0, next_seed!(c), C_NULL, C_NULL, images[r]))
        end
    end
    img = images[1]
    Trace.set_image!(film, [Trace.RGBSpectrum(img[1, x, y], img[2, x, y], img[3, x, y]) for y in 1:H, x in 1:W])
    Trace.save(film)
end
function (g::GPU{Trace.SPPMIntegrator,Context})(scene::Trace.Scene)
    i, ctx = g.integrator, g.ctx
    film = Trace.get_film(i.camera)
    H, W = size(film.pixels)
    rgb = zeros(Float32, 3, W, H)
    function on_image(::Ptr{Cvoid}, iteration::Cint, p::Ptr{Float32})::Cvoid
        img = unsafe_wrap(Array, p, (3, W, H))
        Trace.set_image!(film, [Trace.RGBSpectrum(img[1, x, y], img[2, x, y], img[3, x, y]) for y in 1:H, x in 1:W])
        Trace.save(film)
        nothing
    end
    cb = @cfunction($on_image, Cvoid, (Ptr{Cvoid}, Cint, Ptr{Float32}))
    lock(ctx.lock) do
        upload!(ctx, scene)
        GC.@preserve rgb cb check(ctx, ccall((:trace_render_sppm, LIB), Cint,
            (Ptr{Cvoid}, Ref{CameraP}, Ref{FilmP}, Cfloat, Cint, Cint, Int64, Cint, UInt64, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float32}),
            ctx.h, camera_pod(i.camera), film_pod(film), i.initial_search_radius, i.max_depth, i.n_iterations,
            i.photons_per_iteration, i.write_frequency, next_seed!(ctx), cb, C_NULL, rgb))
    end
end

# batch intersect!(scene, rays) / intersect_p — src/accel/bvh.jl:212-299
function intersect!(ctx::Context, o::Matrix{Float32}, d::Matrix{Float32}, t_max::Vector{Float32})
    n = size(o, 2)
    prim = zeros(UInt32, n); bary = zeros(Float32, 2, n)
    GC.@preserve o d t_max prim bary check(ctx, ccall((:trace_intersect, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float32}, Ptr{Float32}, Ptr{Float32}, Int64, Ptr{UInt32}, Ptr{Float32}),
        ctx.h, o, d, t_max, n, prim, bary))
    prim, bary            # t_max now holds the hit distances, like ray.t_max after intersect!
end


end # module
