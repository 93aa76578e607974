// shading_probe.cu — TEST INFRASTRUCTURE ONLY: batched device calls of the library's own shading functions
// (shading.cuh, wavefront.cuh), so tests can hold them call by call against the CPU oracle.  Built by tests/probe_lib.py
// with the library's NVCCFLAGS and linked against libtrace_cuda.so (ctx_pack_materials and the uploaded scene).
// Every entry point launches one kernel over n inputs and returns 0, or a CUDA error code.
#include "../../trace.jl_b200/csrc/context.hpp"
#include "../../trace.jl_b200/csrc/shading.cuh"
#include "../../trace.jl_b200/csrc/wavefront.cuh"

// the oracle's canonical BSDF frame (oracle/ref_render.cpp canonical_bsdf): ss = x, ns = ng = z, ts = cross(ns, ss)
__device__ __forceinline__ Frame canonical_frame() {
    Frame fr;
    fr.ss = f3(1.0f, 0.0f, 0.0f); fr.ns = f3(0.0f, 0.0f, 1.0f); fr.ng = fr.ns; fr.ts = cross3(fr.ns, fr.ss);
    return fr;
}
__device__ __forceinline__ float3 ld3(const float* p, int i) { return f3(p[3 * i], p[3 * i + 1], p[3 * i + 2]); }
__device__ __forceinline__ void st3(float* p, int k, float3 v) { p[k] = v.x; p[k + 1] = v.y; p[k + 2] = v.z; }

// q[i] = {material index, mode (0 Whitted lobes, 1 SPPM lobes), flags}
__global__ void k_probe_bsdf_f(const DeviceMaterial* mats, const int* q, const float* wo, const float* wi, float* f, int* n_lobes, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    LobeSet s;
    material_lobes(mats[q[3 * i]], q[3 * i + 1] != 0, s);
    st3(f, 3 * i, bsdf_f(s, canonical_frame(), ld3(wo, i), ld3(wi, i), (uint32_t)q[3 * i + 2]));
    n_lobes[i] = s.n;
}

// q[i] = {material index, mode, type}; out[i] = wi(3), f(3), pdf, sampled type (the oracle's ref_bsdf_sample layout)
__global__ void k_probe_bsdf_sample(const DeviceMaterial* mats, const int* q, const float* wo, const float* u, float* out, int* n_lobes, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    LobeSet s;
    material_lobes(mats[q[3 * i]], q[3 * i + 1] != 0, s);
    const BSDFSample b = bsdf_sample(s, canonical_frame(), ld3(wo, i), u[2 * i], u[2 * i + 1], (uint32_t)q[3 * i + 2]);
    st3(out, 8 * i, b.wi);
    st3(out, 8 * i + 3, b.f);
    out[8 * i + 6] = b.pdf;
    out[8 * i + 7] = (float)b.type;
    n_lobes[i] = s.n;
}

// the hit record k_wh_shade builds for BVH slot `slot` hit by ray (o, d) at barycentrics (b0, b1):
// out[i] = p, ng, ns, ss, ts, wo (18 floats); ids[i] = material, original
__global__ void k_probe_hit(DeviceScene sc, const uint32_t* slot, const float* o, const float* d_in, const float* b, float* out,
                            uint32_t* ids, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float3 d = ld3(d_in, i);
    if (d.x == 0.0f) d.x = 0.0f;                        // check_direction!, as k_wh_shade
    if (d.y == 0.0f) d.y = 0.0f;
    if (d.z == 0.0f) d.z = 0.0f;
    const float3 org = ld3(o, i);
    const float b2 = third_barycentric(sc, slot[i], org, d);
    const Interaction it = build_interaction(sc, slot[i], org, d, b[2 * i], b[2 * i + 1], b2);
    const Frame fr = make_frame(it);
    const float3 v[6] = {it.p, it.ng, it.ns, fr.ss, fr.ts, it.wo};
    for (int k = 0; k < 6; ++k) st3(out, 18 * i + 3 * k, v[k]);
    ids[2 * i] = it.material;
    ids[2 * i + 1] = __float_as_uint(__ldg(&sc.prims[3 * slot[i] + 2]).w);
}

__global__ void k_probe_radical_inverse(const int* base_index, const unsigned long long* a, float* out, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = radical_inverse(base_index[i], a[i]);
}

__global__ void k_probe_rng(const uint64_t* seed, const uint32_t* abc, float* out, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = rng_uniform(seed[i], abc[3 * i], abc[3 * i + 1], abc[3 * i + 2]);
}

// device copies of the inputs, the launch, and the copies back; frees everything on every path
namespace {
struct Probe {
    std::vector<void*> bufs;
    cudaError_t err = cudaSuccess;
    ~Probe() { for (void* p : bufs) cudaFree(p); }
    template <class T> T* in(const T* host, size_t count) {
        T* d = out<T>(count);
        if (d && count) note(cudaMemcpy(d, host, count * sizeof(T), cudaMemcpyHostToDevice));
        return d;
    }
    template <class T> T* out(size_t count) {
        void* p = nullptr;
        if (err == cudaSuccess) note(cudaMalloc(&p, count ? count * sizeof(T) : 16));
        if (p) bufs.push_back(p);
        return static_cast<T*>(p);
    }
    template <class T> void back(T* host, const T* dev, size_t count) {
        if (err == cudaSuccess && count) note(cudaMemcpy(host, dev, count * sizeof(T), cudaMemcpyDeviceToHost));
    }
    void note(cudaError_t e) { if (err == cudaSuccess) err = e; }
    void launched() { note(cudaGetLastError()); note(cudaDeviceSynchronize()); }
};
int grid(int64_t n) { return (int)((n + 127) / 128); }
}  // namespace

extern "C" {

// the materials as trace_scene_upload packs them (sigma -> A / B, roughness remap, 1e-3 clamp): -1 when refused
int probe_pack_materials(trace_ctx* c, int64_t n, const trace_material* m, DeviceMaterial* out) {
    std::vector<DeviceMaterial> v;
    if (ctx_pack_materials(c, n, m, v)) return -1;
    for (size_t k = 0; k < v.size(); ++k) out[k] = v[k];
    return 0;
}

int probe_bsdf_f(trace_ctx* c, int64_t n_mat, const trace_material* m, int64_t n, const int* q, const float* wo, const float* wi,
                 float* f, int* n_lobes) {
    std::vector<DeviceMaterial> mats;
    if (ctx_pack_materials(c, n_mat, m, mats)) return -1;
    if (n <= 0) return 0;
    Probe P;
    const DeviceMaterial* dm = P.in(mats.data(), mats.size());
    const int* dq = P.in(q, 3 * n);
    const float *dwo = P.in(wo, 3 * n), *dwi = P.in(wi, 3 * n);
    float* df = P.out<float>(3 * n);
    int* dl = P.out<int>(n);
    if (P.err) return (int)P.err;
    k_probe_bsdf_f<<<grid(n), 128>>>(dm, dq, dwo, dwi, df, dl, (int)n);
    P.launched();
    P.back(f, df, 3 * n);
    P.back(n_lobes, dl, n);
    return (int)P.err;
}

int probe_bsdf_sample(trace_ctx* c, int64_t n_mat, const trace_material* m, int64_t n, const int* q, const float* wo, const float* u,
                      float* out, int* n_lobes) {
    std::vector<DeviceMaterial> mats;
    if (ctx_pack_materials(c, n_mat, m, mats)) return -1;
    if (n <= 0) return 0;
    Probe P;
    const DeviceMaterial* dm = P.in(mats.data(), mats.size());
    const int* dq = P.in(q, 3 * n);
    const float *dwo = P.in(wo, 3 * n), *du = P.in(u, 2 * n);
    float* dout = P.out<float>(8 * n);
    int* dl = P.out<int>(n);
    if (P.err) return (int)P.err;
    k_probe_bsdf_sample<<<grid(n), 128>>>(dm, dq, dwo, du, dout, dl, (int)n);
    P.launched();
    P.back(out, dout, 8 * n);
    P.back(n_lobes, dl, n);
    return (int)P.err;
}

// slots: BVH-ordered primitive slots of the context's uploaded scene
int probe_hit_record(trace_ctx* c, int64_t n, const uint32_t* slot, const float* o, const float* d, const float* b, float* out,
                     uint32_t* ids) {
    if (trace_synchronize(c)) return -1;
    if (!c->have_scene) return -1;
    if (n <= 0) return 0;
    Probe P;
    const uint32_t* ds = P.in(slot, n);
    const float *dorg = P.in(o, 3 * n), *dd = P.in(d, 3 * n), *db = P.in(b, 2 * n);
    float* dout = P.out<float>(18 * n);
    uint32_t* dids = P.out<uint32_t>(2 * n);
    if (P.err) return (int)P.err;
    k_probe_hit<<<grid(n), 128>>>(c->scene, ds, dorg, dd, db, dout, dids, (int)n);
    P.launched();
    P.back(out, dout, 18 * n);
    P.back(ids, dids, 2 * n);
    return (int)P.err;
}

int probe_radical_inverse(int64_t n, const int* base_index, const unsigned long long* a, float* out) {
    if (n <= 0) return 0;
    Probe P;
    const int* db = P.in(base_index, n);
    const unsigned long long* da = P.in(a, n);
    float* dout = P.out<float>(n);
    if (P.err) return (int)P.err;
    k_probe_radical_inverse<<<grid(n), 128>>>(db, da, dout, (int)n);
    P.launched();
    P.back(out, dout, n);
    return (int)P.err;
}

int probe_rng(int64_t n, const uint64_t* seed, const uint32_t* abc, float* out) {
    if (n <= 0) return 0;
    Probe P;
    const uint64_t* ds = P.in(seed, n);
    const uint32_t* dabc = P.in(abc, 3 * n);
    float* dout = P.out<float>(n);
    if (P.err) return (int)P.err;
    k_probe_rng<<<grid(n), 128>>>(ds, dabc, dout, (int)n);
    P.launched();
    P.back(out, dout, n);
    return (int)P.err;
}

}  // extern "C"
