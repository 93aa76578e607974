// bvh_gpu.cu — opt-in LBVH build on the GPU (trace_bvh_build_gpu, include/trace_cuda.h).
//
// A Karras (2012) binary radix tree over 63-bit Morton codes of the primitive centroids, emitted in the same flattened
// preorder node format as the host builders (first child = parent + 1), so every kernel walks it unchanged.  The tree
// is fully specified by its inputs (tests/test_gpu_lbvh.py restates it in numpy and compares bit for bit):
//   centroid   c = 0.5 bmin + 0.5 bmax (the host builders' formula), float32, unfused (-fmad=false);
//   quantised  q = min(2^21 - 1, floor((c - lo) * s)) with s = 2^21 / (hi - lo) per axis (0 for a flat axis), lo / hi
//              the exact centroid box;
//   key        x at bit 3k+2, y at 3k+1, z at 3k; sorted stably, so the order is lexicographic on (key, index);
//   split      at the highest bit where the range's first and last key differ (left child: that bit 0, axis 2 - h % 3),
//              or, for a range of equal keys, at the highest differing bit of the two positions (axis 0);
//   leaf       a range of <= max_node_primitives primitives (its whole subtree collapses into one node).
// Node boxes use Julia's min / max (-0.0 < +0.0): with NaN refused the union is exact and independent of the order in
// which the bottom-up threads arrive, so the output is deterministic.
#include <algorithm>
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>

#include <cub/device/device_radix_sort.cuh>

#include "../../include/trace_cuda.h"

// bvh_build.cpp: an uninitialised host handle with room for the given arrays (nullptr when out of memory)
trace_bvh* bvh_alloc(int64_t n_nodes, int64_t n_prims, trace_bvh_node** nodes, uint32_t** order);

namespace {

// Node ids: internal nodes 0 .. n-2 (Karras numbering), leaf k (sorted position k) is n-1+k.  The root is id 0 in both
// cases (n == 1: the single leaf).
struct Status {
    uint32_t cmin[3], cmax[3];      // centroid box as order-preserving keys (ord_key)
    uint32_t nan;                   // a centroid is NaN
    uint32_t root_size, root_depth; // emitted nodes, levels (root = 1)
    uint32_t bad;                   // mesh builds: a NaN normal (bit 0), a material index out of range (bit 1)
};

// float <-> uint32 in Julia's total order on non-NaN floats (-0.0 sorts below +0.0), so atomicMin / atomicMax pick it
__device__ __forceinline__ uint32_t ord_key(float f) {
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord_float(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}
// Julia's min / max without NaN: exact, and -0.0 < +0.0
__device__ __forceinline__ float jl_min(float a, float b) { return (b < a || (b == a && signbit(b))) ? b : a; }
__device__ __forceinline__ float jl_max(float a, float b) { return (b > a || (b == a && !signbit(b))) ? b : a; }

__device__ __forceinline__ float centroid(const float* pb, int64_t i, int k) {
    return __fadd_rn(__fmul_rn(0.5f, pb[6 * i + k]), __fmul_rn(0.5f, pb[6 * i + 3 + k]));
}

// 21 bits -> every third bit of 63
__device__ __forceinline__ uint64_t spread3(uint64_t x) {
    x &= 0x1FFFFFull;
    x = (x | x << 32) & 0x1F00000000FFFFull;
    x = (x | x << 16) & 0x1F0000FF0000FFull;
    x = (x | x << 8) & 0x100F00F00F00F00Full;
    x = (x | x << 4) & 0x10C30C30C30C30C3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}

// 1. exact centroid box (Julia order) and the NaN flag
__global__ void lbvh_centroid_box(const float* __restrict__ pb, int64_t n, Status* st) {
    uint32_t lo[3] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu}, hi[3] = {0u, 0u, 0u};
    bool nan = false;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        for (int k = 0; k < 3; ++k) {
            const float c = centroid(pb, i, k);
            if (c != c) { nan = true; continue; }
            const uint32_t q = ord_key(c);
            lo[k] = min(lo[k], q);
            hi[k] = max(hi[k], q);
        }
    }
    for (int k = 0; k < 3; ++k) {
        lo[k] = __reduce_min_sync(0xFFFFFFFFu, lo[k]);
        hi[k] = __reduce_max_sync(0xFFFFFFFFu, hi[k]);
    }
    nan = __any_sync(0xFFFFFFFFu, nan);
    if ((threadIdx.x & 31) == 0) {
        for (int k = 0; k < 3; ++k) { atomicMin(&st->cmin[k], lo[k]); atomicMax(&st->cmax[k], hi[k]); }
        if (nan) atomicOr(&st->nan, 1u);
    }
}

// 2. Morton keys and the identity permutation (the sort's values)
__global__ void lbvh_keys(const float* __restrict__ pb, int64_t n, const Status* __restrict__ st, uint64_t* __restrict__ keys,
                          uint32_t* __restrict__ ids) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t key = 0;
    for (int k = 0; k < 3; ++k) {
        const float lo = ord_float(st->cmin[k]), hi = ord_float(st->cmax[k]);
        const float ext = __fsub_rn(hi, lo);
        const float s = ext > 0.0f ? __fdiv_rn(2097152.0f, ext) : 0.0f;
        const float v = __fmul_rn(__fsub_rn(centroid(pb, i, k), lo), s);
        // v >= 0 (c >= lo); a NaN (0 * inf on a denormal-thin axis) is position 0
        const uint32_t q = v >= 2097151.0f ? 2097151u : (v > 0.0f ? (uint32_t)floorf(v) : 0u);
        key |= spread3(q) << (2 - k);
    }
    keys[i] = key;
    ids[i] = (uint32_t)i;
}

// common prefix length of the strings (key, position) at sorted positions i and j; -1 outside [0, n)
__device__ __forceinline__ int delta(const uint64_t* __restrict__ K, int64_t n, int64_t i, int64_t j) {
    if (j < 0 || j >= n) return -1;
    const uint64_t a = K[i], b = K[j];
    if (a != b) return __clzll((long long)(a ^ b));
    return 64 + __clz((int)((uint32_t)i ^ (uint32_t)j));
}

// 3. hierarchy: internal node i finds its range and split (Karras 2012, Fig. 4)
__global__ void lbvh_hierarchy(const uint64_t* __restrict__ K, int64_t n, uint32_t* __restrict__ child,
                               int32_t* __restrict__ parent, uint32_t* __restrict__ first, uint32_t* __restrict__ count,
                               uint8_t* __restrict__ axis) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    const int d = delta(K, n, i, i + 1) - delta(K, n, i, i - 1) > 0 ? 1 : -1;
    const int dmin = delta(K, n, i, i - d);
    int64_t lmax = 2;
    while (delta(K, n, i, i + lmax * d) > dmin) lmax *= 2;
    int64_t l = 0;
    for (int64_t t = lmax / 2; t >= 1; t /= 2)
        if (delta(K, n, i, i + (l + t) * d) > dmin) l += t;
    const int64_t j = i + l * d;
    const int dnode = delta(K, n, i, j);
    int64_t s = 0;
    for (int64_t div = 2;; div *= 2) {
        const int64_t t = (l + div - 1) / div;
        if (delta(K, n, i, i + (s + t) * d) > dnode) s += t;
        if (t == 1) break;
    }
    const int64_t gamma = i + s * d + (d < 0 ? -1 : 0);
    const int64_t lo = d > 0 ? i : j, hi = d > 0 ? j : i;
    const uint32_t left = (uint32_t)(lo == gamma ? (n - 1) + gamma : gamma);
    const uint32_t right = (uint32_t)(hi == gamma + 1 ? (n - 1) + gamma + 1 : gamma + 1);
    child[2 * i] = left;
    child[2 * i + 1] = right;
    parent[left] = (int32_t)i;
    parent[right] = (int32_t)i;
    first[i] = (uint32_t)lo;
    count[i] = (uint32_t)(hi - lo + 1);
    const uint64_t x = K[lo] ^ K[hi];
    axis[i] = x ? (uint8_t)(2 - (63 - __clzll((long long)x)) % 3) : 0;
}

// 4. bottom-up: boxes, emitted subtree sizes and depths; one thread per leaf climbs while it is the second to arrive
__global__ void lbvh_bottom_up(const float* __restrict__ pb, const uint32_t* __restrict__ sorted_ids, int64_t n, int m,
                               const uint32_t* __restrict__ child, const int32_t* __restrict__ parent,
                               const uint32_t* __restrict__ count, uint32_t* arrive, float* box, uint32_t* size,
                               uint32_t* depth, Status* st) {
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= n) return;
    int64_t v = (n - 1) + k;
    const int64_t p0 = sorted_ids[k];
    for (int c = 0; c < 6; ++c) box[6 * v + c] = pb[6 * p0 + c];
    size[v] = 1;
    depth[v] = 1;
    for (;;) {
        const int32_t p = parent[v];
        if (p < 0) break;
        __threadfence();
        if (atomicAdd(&arrive[p], 1u) == 0) return;           // the sibling's thread continues
        __threadfence();
        const uint32_t l = child[2 * p], r = child[2 * p + 1];
        for (int c = 0; c < 3; ++c) {
            box[6 * (int64_t)p + c] = jl_min(__ldcg(&box[6 * (int64_t)l + c]), __ldcg(&box[6 * (int64_t)r + c]));
            box[6 * (int64_t)p + 3 + c] = jl_max(__ldcg(&box[6 * (int64_t)l + 3 + c]), __ldcg(&box[6 * (int64_t)r + 3 + c]));
        }
        const bool leaf = count[p] <= (uint32_t)m;
        size[p] = leaf ? 1u : 1u + __ldcg(&size[l]) + __ldcg(&size[r]);
        depth[p] = leaf ? 1u : 1u + max(__ldcg(&depth[l]), __ldcg(&depth[r]));
        v = p;
    }
    st->root_size = size[0];                                 // v == 0: the last thread to arrive at the root
    st->root_depth = depth[0];
}

// 5. emit: every emitted node finds its preorder slot by climbing to the root (left child = parent + 1, right child =
// parent + 1 + size(left); depth <= TR_STACK_SIZE is checked before this runs) and writes its record
__global__ void lbvh_emit(int64_t n, int m, const uint32_t* __restrict__ child, const int32_t* __restrict__ parent,
                          const uint32_t* __restrict__ first, const uint32_t* __restrict__ count,
                          const uint8_t* __restrict__ axis, const float* __restrict__ box, const uint32_t* __restrict__ size,
                          trace_bvh_node* __restrict__ out) {
    const int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v >= 2 * n - 1) return;
    const bool internal = v < n - 1;
    const int32_t pv = parent[v];
    if (pv >= 0 && count[pv] <= (uint32_t)m) return;         // inside a collapsed subtree
    uint32_t pre = 0;
    for (int64_t c = v; c != 0;) {
        const int32_t p = parent[c];
        const uint32_t l = child[2 * p];
        pre += c == l ? 1u : 1u + size[l];
        c = p;
    }
    trace_bvh_node nd;
    for (int c = 0; c < 3; ++c) { nd.bmin[c] = box[6 * v + c]; nd.bmax[c] = box[6 * v + 3 + c]; }
    const uint32_t cnt = internal ? count[v] : 1u;
    if (cnt <= (uint32_t)m) {
        nd.offset = internal ? first[v] : (uint32_t)(v - (n - 1));
        nd.meta = TRACE_NODE_LEAF | cnt;
    } else {
        nd.offset = pre + 1u + size[child[2 * v]];
        nd.meta = (uint32_t)axis[v] << 30;
    }
    out[pre] = nd;
}

inline unsigned blocks_for(int64_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }

// The build's device buffers, carved out of one allocation: carve() with base == 0 sizes it, then again on the real one.
// `pb` (the primitive bounds) and the node array are carved only when asked for.
struct Buffers {
    float* pb = nullptr; Status* st;
    uint64_t *keys, *keys_sorted; uint32_t *ids, *ids_sorted;                  // sort in / out
    uint32_t *child, *first, *count; int32_t* parent; uint8_t* axis;           // hierarchy (parent: every node)
    uint32_t* arrive; float* box; uint32_t *size, *depth;                      // bottom-up, every node
    trace_bvh_node* nodes = nullptr; void* sort_tmp;
    size_t used = 0;
    char* base = nullptr;
    template <class T> T* take(int64_t count) {
        const size_t off = (used + 255) & ~(size_t)255;
        used = off + (size_t)count * sizeof(T);
        return reinterpret_cast<T*>(base + off);
    }
    void carve(int64_t n, size_t sort_bytes, bool with_pb, bool with_nodes) {
        const int64_t nn = 2 * n - 1;
        used = 0;
        if (with_pb) pb = take<float>(6 * n);
        st = take<Status>(1);
        keys = take<uint64_t>(n); keys_sorted = take<uint64_t>(n); ids = take<uint32_t>(n); ids_sorted = take<uint32_t>(n);
        child = take<uint32_t>(2 * (n - 1)); first = take<uint32_t>(n - 1); count = take<uint32_t>(n - 1);
        parent = take<int32_t>(nn); axis = take<uint8_t>(n - 1);
        arrive = take<uint32_t>(n - 1); box = take<float>(6 * nn); size = take<uint32_t>(nn); depth = take<uint32_t>(nn);
        if (with_nodes) nodes = take<trace_bvh_node>(nn);
        sort_tmp = take<char>((int64_t)sort_bytes);
    }
    // one allocation for everything; freed by the destructor
    int alloc(int64_t n, size_t sort_bytes, bool with_pb, bool with_nodes) {
        carve(n, sort_bytes, with_pb, with_nodes);
        if (cudaMalloc(&base, used) != cudaSuccess) { cudaGetLastError(); base = nullptr; return 7; }
        owned = true;
        carve(n, sort_bytes, with_pb, with_nodes);
        return 0;
    }
    // the caller's allocation of at least lbvh_scratch_bytes(n) bytes (with pb, without nodes); kept by the caller
    void borrow(void* scratch, int64_t n, size_t sort_bytes) {
        base = static_cast<char*>(scratch);
        carve(n, sort_bytes, true, false);
    }
    bool owned = false;
    ~Buffers() { if (owned) cudaFree(base); }
};

struct Phases {
    bool on = false;
    cudaEvent_t ev[8] = {};
    int n = 0;
    void mark(cudaStream_t s) { if (on && n < 8) cudaEventRecord(ev[n++], s); }
};

size_t sort_bytes_for(int64_t n, cudaStream_t s) {
    size_t bytes = 0;
    if (cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const uint32_t*)nullptr,
                                        (uint32_t*)nullptr, (int)n, 0, 63, s) != cudaSuccess)
        return 0;
    return bytes;
}

// The device-resident core: bounds b.pb (device, [n][6]) -> keys, sorted order, hierarchy, boxes, subtree sizes and
// depths in `b`, and the status on the host.  Returns 0, 5 (a NaN bound), 6 (deeper than the 64-entry traversal
// stack) or 7 (CUDA error).
void core_reset(cudaStream_t s, int64_t n, Buffers& b) {
    cudaMemsetAsync(b.st, 0xFF, sizeof(b.st->cmin), s);
    cudaMemsetAsync(&b.st->cmax, 0, sizeof(Status) - sizeof(b.st->cmin), s);
    cudaMemsetAsync(b.parent, 0xFF, (size_t)(2 * n - 1) * sizeof(int32_t), s);
    if (n > 1) cudaMemsetAsync(b.arrive, 0, (size_t)(n - 1) * sizeof(uint32_t), s);
}

// build_core without the reset: what runs after core_reset (and anything that reports into the status block)
int core_run(cudaStream_t s, int64_t n, int m, Buffers& b, size_t sort_bytes, Status& hs, Phases& ph) {
    const int T = 256;
    lbvh_centroid_box<<<(unsigned)std::min<int64_t>(blocks_for(n, T), 4096), T, 0, s>>>(b.pb, n, b.st);
    lbvh_keys<<<blocks_for(n, T), T, 0, s>>>(b.pb, n, b.st, b.keys, b.ids);
    ph.mark(s);
    if (cub::DeviceRadixSort::SortPairs(b.sort_tmp, sort_bytes, b.keys, b.keys_sorted, b.ids, b.ids_sorted, (int)n, 0, 63, s)
        != cudaSuccess)
        return 7;
    ph.mark(s);
    if (n > 1) lbvh_hierarchy<<<blocks_for(n - 1, T), T, 0, s>>>(b.keys_sorted, n, b.child, b.parent, b.first, b.count, b.axis);
    ph.mark(s);
    lbvh_bottom_up<<<blocks_for(n, T), T, 0, s>>>(b.pb, b.ids_sorted, n, m, b.child, b.parent, b.count, b.arrive, b.box,
                                                   b.size, b.depth, b.st);
    if (cudaGetLastError() != cudaSuccess ||
        cudaMemcpyAsync(&hs, b.st, sizeof(Status), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
        cudaStreamSynchronize(s) != cudaSuccess)
        return 7;
    ph.mark(s);
    if (hs.nan) return 5;
    if (hs.root_depth > 64) return 6;                        // TR_STACK_SIZE (traverse.cuh): the walks' stacks would overflow
    return 0;
}

int build_core(cudaStream_t s, int64_t n, int m, Buffers& b, size_t sort_bytes, Status& hs, Phases& ph) {
    core_reset(s, n, b);
    return core_run(s, n, m, b, sort_bytes, hs, ph);
}

int build(cudaStream_t s, const float* hb, int64_t n, int m, trace_bvh** out, Phases& ph) {
    const int64_t nn = 2 * n - 1;
    const size_t sort_bytes = sort_bytes_for(n, s);
    if (!sort_bytes) return 7;
    Buffers b;
    if (b.alloc(n, sort_bytes, true, true)) return 7;
    const int T = 256;
    ph.mark(s);
    if (cudaMemcpyAsync(b.pb, hb, (size_t)n * 6 * sizeof(float), cudaMemcpyHostToDevice, s) != cudaSuccess) return 7;
    ph.mark(s);
    Status hs;
    if (const int rc = build_core(s, n, m, b, sort_bytes, hs, ph)) return rc;
    const int64_t n_nodes = hs.root_size;
    lbvh_emit<<<blocks_for(nn, T), T, 0, s>>>(n, m, b.child, b.parent, b.first, b.count, b.axis, b.box, b.size, b.nodes);
    if (cudaGetLastError() != cudaSuccess) return 7;
    ph.mark(s);
    trace_bvh_node* hn = nullptr;
    uint32_t* ho = nullptr;
    trace_bvh* bvh = bvh_alloc(n_nodes, n, &hn, &ho);
    if (!bvh) return 2;
    if (cudaMemcpyAsync(hn, b.nodes, (size_t)n_nodes * sizeof(trace_bvh_node), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
        cudaMemcpyAsync(ho, b.ids_sorted, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost, s) != cudaSuccess) {
        trace_bvh_free(bvh);
        return 7;
    }
    ph.mark(s);
    if (cudaStreamSynchronize(s) != cudaSuccess) { trace_bvh_free(bvh); return 7; }
    *out = bvh;
    return 0;
}

// ------------------------------------------------------------------ the shadow tree (traverse.cuh, traverse_shadow)
// A primitive's box: Julia min / max over its three vertices (the refit's leaf rule, refit.cu).  A NaN coordinate makes
// the whole box NaN, so the centroid pass refuses the input.
__global__ void lbvh_prim_bounds(const float4* __restrict__ prims, int64_t n, float* __restrict__ pb) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 A = prims[3 * i], B = prims[3 * i + 1], C = prims[3 * i + 2];
    float lo[3] = {jl_min(jl_min(jl_min(INFINITY, A.x), B.x), C.x), jl_min(jl_min(jl_min(INFINITY, A.y), B.y), C.y),
                   jl_min(jl_min(jl_min(INFINITY, A.z), B.z), C.z)};
    float hi[3] = {jl_max(jl_max(jl_max(-INFINITY, A.x), B.x), C.x), jl_max(jl_max(jl_max(-INFINITY, A.y), B.y), C.y),
                   jl_max(jl_max(jl_max(-INFINITY, A.z), B.z), C.z)};
    const bool nan = A.x != A.x || A.y != A.y || A.z != A.z || B.x != B.x || B.y != B.y || B.z != B.z || C.x != C.x ||
                     C.y != C.y || C.z != C.z;
    for (int c = 0; c < 3; ++c) {
        pb[6 * i + c] = nan ? NAN : lo[c];
        pb[6 * i + 3 + c] = nan ? NAN : hi[c];
    }
}

// One 64-byte pair record per internal node, in Karras numbering (the root is pair 0): both children's boxes, their
// references (a pair index, or 0x80000000 | primitive slot for a leaf: TR_REF_LEAF, traverse.cuh) and the split axis as
// a bit in the first half - the layout of the upload's pair records (api.cu).
__global__ void lbvh_emit_pairs(int64_t n, const uint32_t* __restrict__ child, const uint32_t* __restrict__ sorted_ids,
                                const uint8_t* __restrict__ axis, const float* __restrict__ box, float4* __restrict__ pairs) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    for (int k = 0; k < 2; ++k) {
        const int64_t v = child[2 * i + k];
        const float* bx = box + 6 * v;
        const uint32_t ref = v < n - 1 ? (uint32_t)v : (0x80000000u | sorted_ids[v - (n - 1)]);
        const uint32_t extra = k == 0 ? (1u << axis[i]) : 0u;
        pairs[4 * i + 2 * k] = make_float4(bx[0], bx[1], bx[2], bx[3]);
        pairs[4 * i + 2 * k + 1] = make_float4(bx[4], bx[5], __uint_as_float(ref), __uint_as_float(extra));
    }
}

// ------------------------------------------------------------------ mesh builds (trace_scene_upload_mesh_device, upload_device.cu)
// The inputs a triangle array brings beyond its vertices: any NaN normal (bit 0) and any material index >= n_materials
// (bit 1) into the status block, which the build reads back before anything is emitted.
__global__ void lbvh_mesh_validate(const float* __restrict__ nrm, const uint32_t* __restrict__ mat, int64_t n,
                                   uint32_t n_materials, Status* st) {
    uint32_t bad = 0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (nrm)
            for (int k = 0; k < 9; ++k) { const float x = nrm[9 * i + k]; if (x != x) bad |= 1u; }
        if ((mat ? mat[i] : 0u) >= n_materials) bad |= 2u;
    }
    bad = __reduce_or_sync(0xFFFFFFFFu, bad);
    if ((threadIdx.x & 31) == 0 && bad) atomicOr(&st->bad, bad);
}

// A triangle's box from the [n][3][3] vertex array: the rule of lbvh_prim_bounds (a NaN vertex makes the box NaN)
__global__ void lbvh_tri_bounds(const float* __restrict__ v, int64_t n, float* __restrict__ pb) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* p = v + 9 * i;
    bool nan = false;
    for (int k = 0; k < 9; ++k) nan |= p[k] != p[k];
    for (int c = 0; c < 3; ++c) {
        pb[6 * i + c] = nan ? NAN : jl_min(jl_min(jl_min(INFINITY, p[c]), p[3 + c]), p[6 + c]);
        pb[6 * i + 3 + c] = nan ? NAN : jl_max(jl_max(jl_max(-INFINITY, p[c]), p[3 + c]), p[6 + c]);
    }
}

}  // namespace

// Scratch of one LBVH build over n primitives (bounds, keys, sort, hierarchy, boxes) in a caller-owned allocation;
// 0 when CUB cannot size its sort.  The shadow tree's build of the same n fits the same bytes.
size_t lbvh_scratch_bytes(int64_t n, cudaStream_t s) {
    const size_t sort_bytes = sort_bytes_for(n, s);
    if (!sort_bytes) return 0;
    Buffers b;
    b.carve(n, sort_bytes, true, false);
    return b.used;
}

// The shadow tree of an uploaded scene (api.cu): an LBVH with one primitive per leaf over the n >= 2 uploaded primitive
// records `prims` (device, BVH slot order, triangles only), written as n - 1 pair records to `pairs` (device).  Nothing
// crosses to the host but the build's status.  `scratch` (lbvh_scratch_bytes(n)) or nullptr: an allocation of its own.
// Returns 0, 5 (a NaN vertex), 6 (deeper than 64 levels) or 7 (CUDA error).
int shadow_tree_build(cudaStream_t s, const void* prims, int64_t n, void* pairs, void* scratch) {
    if (n < 2 || n >= 0x40000000ll) return 1;
    const size_t sort_bytes = sort_bytes_for(n, s);
    if (!sort_bytes) return 7;
    Buffers b;
    if (scratch) b.borrow(scratch, n, sort_bytes);
    else if (b.alloc(n, sort_bytes, true, false)) return 7;
    const int T = 256;
    lbvh_prim_bounds<<<blocks_for(n, T), T, 0, s>>>(static_cast<const float4*>(prims), n, b.pb);
    Phases ph;
    Status hs;
    if (const int rc = build_core(s, n, 1, b, sort_bytes, hs, ph)) return rc;
    lbvh_emit_pairs<<<blocks_for(n - 1, T), T, 0, s>>>(n, b.child, b.ids_sorted, b.axis, b.box, static_cast<float4*>(pairs));
    if (cudaGetLastError() != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess) return 7;
    return 0;
}

// The tree of trace_scene_upload_mesh_device, in steps over `scratch` (lbvh_scratch_bytes(n), n >= 1):
//   lbvh_mesh_validate  reset the status block, check normals (NULL: none) and material indices (NULL: all 0) into it;
//   lbvh_mesh_bounds    the triangles' boxes (no host wait so far);
//   lbvh_mesh_build     the LBVH core and its status read back: 0, 5 a NaN vertex, 6 deeper than 64 levels, 7 CUDA
//                       error, 8 a NaN normal, 9 a material index out of range; *n_nodes, and *order = the sorted
//                       triangle ids (slot -> triangle, device, inside the scratch);
//   lbvh_mesh_emit      the preorder node records (trace_bvh_node, 32 B) into `nodes` (device).
// Nothing is written outside the scratch before lbvh_mesh_emit, so a refused input leaves the caller's buffers intact.
int lbvh_mesh_validate(cudaStream_t s, const float* nrm, const uint32_t* mat, int64_t n_materials, int64_t n, void* scratch) {
    const size_t sort_bytes = sort_bytes_for(n, s);
    if (!sort_bytes) return 7;
    Buffers b;
    b.borrow(scratch, n, sort_bytes);
    core_reset(s, n, b);
    const int T = 256;
    const uint32_t nm = n_materials > 0xFFFFFFFFll ? 0xFFFFFFFFu : (uint32_t)n_materials;
    lbvh_mesh_validate<<<(unsigned)std::min<int64_t>(blocks_for(n, T), 4096), T, 0, s>>>(nrm, mat, n, nm, b.st);
    return cudaGetLastError() == cudaSuccess ? 0 : 7;
}

int lbvh_mesh_bounds(cudaStream_t s, const float* v, int64_t n, void* scratch) {
    const size_t sort_bytes = sort_bytes_for(n, s);
    if (!sort_bytes) return 7;
    Buffers b;
    b.borrow(scratch, n, sort_bytes);
    const int T = 256;
    lbvh_tri_bounds<<<blocks_for(n, T), T, 0, s>>>(v, n, b.pb);
    return cudaGetLastError() == cudaSuccess ? 0 : 7;
}

int lbvh_mesh_build(cudaStream_t s, int64_t n, int m, void* scratch, int64_t* n_nodes, const uint32_t** order) {
    const size_t sort_bytes = sort_bytes_for(n, s);
    if (!sort_bytes) return 7;
    Buffers b;
    b.borrow(scratch, n, sort_bytes);
    Phases ph;
    Status hs;
    const int rc = core_run(s, n, m, b, sort_bytes, hs, ph);
    if (rc == 7) return 7;
    if (hs.nan) return 5;                  // the order of the refusals: vertices, normals, materials, depth
    if (hs.bad & 1u) return 8;
    if (hs.bad & 2u) return 9;
    if (rc) return rc;
    *n_nodes = hs.root_size;
    *order = b.ids_sorted;
    return 0;
}

int lbvh_mesh_emit(cudaStream_t s, int64_t n, int m, void* scratch, void* nodes) {
    const size_t sort_bytes = sort_bytes_for(n, s);
    if (!sort_bytes) return 7;
    Buffers b;
    b.borrow(scratch, n, sort_bytes);
    const int T = 256;
    lbvh_emit<<<blocks_for(2 * n - 1, T), T, 0, s>>>(n, m, b.child, b.parent, b.first, b.count, b.axis, b.box, b.size,
                                                    static_cast<trace_bvh_node*>(nodes));
    return cudaGetLastError() == cudaSuccess ? 0 : 7;
}

extern "C" int trace_bvh_build_gpu(int device, const float* pb, int64_t n, int max_node_primitives, trace_bvh** out) {
    if (!out || n < 0 || (n > 0 && !pb)) return 1;
    *out = nullptr;
    if (n >= 0x40000000ll) return 1;
    const int m = max_node_primitives < 1 ? 1 : (max_node_primitives < 255 ? max_node_primitives : 255);
    int n_dev = 0, prev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || device < 0 || device >= n_dev || cudaGetDevice(&prev) != cudaSuccess) {
        cudaGetLastError();
        return 7;                                            // no CPU fallback
    }
    if (n == 0) {
        trace_bvh_node* hn; uint32_t* ho;
        *out = bvh_alloc(0, 0, &hn, &ho);
        return *out ? 0 : 2;
    }
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return 7; }
    cudaStream_t s;
    int rc = 7;
    if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) == cudaSuccess) {
        Phases ph;
        ph.on = getenv("TRACE_BVH_PROFILE") != nullptr;
        for (int i = 0; ph.on && i < 8; ++i) cudaEventCreate(&ph.ev[i]);
        const auto t0 = std::chrono::steady_clock::now();
        rc = build(s, pb, n, m, out, ph);
        if (ph.on && rc == 0) {
            const double wall = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
            static const char* names[7] = {"upload", "keys", "sort", "hierarchy", "bottom-up", "emit", "download"};
            fprintf(stderr, "bvh build gpu: n %lld, device %d, wall %.3f ms;", (long long)n, device, wall);
            for (int i = 0; i + 1 < ph.n; ++i) {
                float ms = 0.0f;
                cudaEventElapsedTime(&ms, ph.ev[i], ph.ev[i + 1]);
                fprintf(stderr, " %s %.3f ms%s", names[i], ms, i + 2 < ph.n ? "," : "\n");
            }
        }
        for (int i = 0; ph.on && i < 8; ++i) cudaEventDestroy(ph.ev[i]);
        cudaStreamDestroy(s);
    }
    cudaGetLastError();
    cudaSetDevice(prev);
    return rc;
}
